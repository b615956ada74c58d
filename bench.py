#!/usr/bin/env python
"""bench.py -- simulated events/sec on the BASELINE workload.

Workload (config.workload): R independent replicas per GPU of the 100k-job
synthetic trace (SURVEY 8d generator, distinct seeds) on the 4x32x8 cluster,
fifo policy + yarn placement -- the only policy/scheme pair the reference can
execute (SURVEY section 0) and therefore the one with a pinned bit-exact oracle.
One "step" = one full simulation of every replica (one persistent-kernel
launch, one warp per replica).  A single replica is latency bound by
construction (<= 1 placement per simulated tick), so throughput comes from
replicas -- the sweeps the reference's execute.py runs serially.

  value  : events/s with traces resident in HBM (device-timed with CUDA events
           around the engine kernel + state reset, max over ranks)
  e2e    : events/s through the C ABI with HOST buffers: every step re-uploads
           every trace (pinned staging -> H2D) and reads back every statistics
           row, job record, finish order and placement span (D2H)
  impl=reference : the CPU oracle port (oracle/gsched_oracle.c, a restatement of
           the reference's Python loop) on all host cores, one replica per thread

Launch:  python bench.py --gpus N --steps K --warmup W   (torchrun for N > 1)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
# The tree the benchmark runs from may be read-only: no bytecode caches in it, from this process or the ones it starts.
# Whatever else it builds goes to a temporary directory.
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

METRIC = "simulated events/sec (100k-job trace, 4x32x8 cluster)"
# --config: c1 = the BASELINE metric's configuration (default); c5 = BASELINE configs[4]: 16x64x8 cluster, 1M-job trace
# (arrivals 8x faster because the cluster is 8x larger; at most one fifo job starts per tick, so this is the deep-queue regime)
CONFIGS = {"c1": dict(num_switch=4, num_node_p_switch=32, jobs=100000, rate=0.5, replicas=4144, label="4x32x8",
                      metric=METRIC),
           "c5": dict(num_switch=16, num_node_p_switch=64, jobs=1000000, rate=4.0, replicas=296, label="16x64x8",
                      metric="simulated events/sec (1M-job trace, 16x64x8 cluster)")}


def apply_config(args):
    cfg = CONFIGS[args.config]
    if args.jobs is None:
        args.jobs = cfg["jobs"]
    if args.replicas is None:
        args.replicas = cfg["replicas"]
    return cfg
UNIT = "events/s"
BASE_SEED = 1


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def fast_table(n_jobs, seed, rate=0.5):
    """Synthetic columns -> JobTable without the pandas round trip (rows are generated in
    arrival order already; only tie order inside a tick differs from a CSV ingest)."""
    from gpuschedule_b200 import ingest, tracegen
    c = tracegen.synth_columns(n_jobs, seed=seed, rate=rate)
    nt = c["normalized_time"].astype(np.float64) / 10000.0
    return ingest.JobTable(
        n=n_jobs, label=None, num_gpu_text=None,
        arrive_tick=np.ceil(nt).astype(np.int32), submit=nt.astype(np.int32),
        gpus=c["used_gpus"].astype(np.int32), gpu_per_task=c["gpu_per_container"].astype(np.int32),
        duration=np.ascontiguousarray(c["minutes"] * 0.5), mem_bytes=c["memory_max"].astype(np.int64),
        util_avg=c["gpu_utilization_avg"], util_max=c["gpu_utilization_max"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def run_to_done(eng, rows_cap, totals=None):
    """run every replica to its end; `totals` (dict) receives per replica the records written over ALL windows"""
    while True:
        eng.run(0, rows_cap)
        if totals is not None:
            for s in range(eng.nsims):
                w = eng.window(s)
                t = totals.setdefault(s, [0, 0])
                t[0] += int(w.ev_rows); t[1] += int(w.q_rows)
        if all(eng.stats(s).done for s in range(eng.nsims)):
            return


DUMP_SEED = 0
DUMP_REPLICAS, DUMP_JOBS, DUMP_ROWS = 3, 100000, 4096      # 43 MB on the c1 workload
DUMP_LIMIT = 64 << 20


def dump_outputs(eng, out_dir):
    """Write what the last timed step computed, as the engine's caller receives it (gs_stats, gs_window, gs_fetch_rows,
    gs_fetch_jobs, gs_fetch_spans), to out_dir/<name>.npy: 2-D float64 tables whose first column is the replica.
    The samples are drawn with a fixed seed, so two builds run with the same arguments write comparable files.

      replica_stats : every replica: ticks, events, finished, started, placement_evals, done,
                      ev_rows, q_rows, node_events, spans_used, admitted
      jobs          : DUMP_REPLICAS sampled replicas x up to DUMP_JOBS sampled jobs: job, start, end, jct, preempt, duration
      finish_order  : the same replicas, up to DUMP_JOBS sampled positions: position, job
      spans         : the placement spans of the sampled jobs: job, node, ntasks, devmask
      rows          : the same replicas, up to DUMP_ROWS sampled statistics rows (the last one always): the gs_tick_row fields
    """
    from gpuschedule_b200.log_manager import ROW_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(DUMP_SEED)
    R = eng.nsims
    stat_f = ("ticks", "events", "finished", "started", "placement_evals", "done")
    win_f = ("ev_rows", "q_rows", "node_events", "spans_used", "admitted")
    stats = np.zeros((R, 1 + len(stat_f) + len(win_f)))
    for r in range(R):
        st, w = eng.stats(r), eng.window(r)
        stats[r] = [r] + [getattr(st, f) for f in stat_f] + [getattr(w, f) for f in win_f]

    def pick(count, cap):
        return np.arange(count) if count <= cap else np.sort(rng.choice(count, size=cap, replace=False))

    row_f = [f for f in ROW_DTYPE.names if f != "reserved"]
    jobs, order, spans, rows = [], [], [], []
    for r in pick(R, DUMP_REPLICAS):
        r = int(r)
        recs, fin = eng.fetch_jobs(r)
        off, sp = eng.fetch_spans(r)
        j = pick(len(recs), DUMP_JOBS)
        jobs.append(np.column_stack([np.full(len(j), r), j] + [recs[f][j] for f in recs.dtype.names]))
        p = pick(len(fin), DUMP_JOBS)
        order.append(np.column_stack([np.full(len(p), r), p, fin[p]]))
        cnt = off[j + 1] - off[j]
        s = np.repeat(off[j] - (np.cumsum(cnt) - cnt), cnt) + np.arange(cnt.sum())      # the spans of job j[i] in order
        spans.append(np.column_stack([np.full(len(s), r), np.repeat(j, cnt), sp["node"][s], sp["ntasks"][s], sp["devmask"][s]]))
        tr = eng.fetch_rows(r, int(eng.window(r).row_first))
        k = np.union1d(pick(len(tr), DUMP_ROWS - 1), [len(tr) - 1]) if len(tr) else np.zeros(0, dtype=np.int64)
        rows.append(np.column_stack([np.full(len(k), r)] + [tr[f][k] for f in row_f]))
    out = {"replica_stats": stats, "jobs": np.concatenate(jobs), "finish_order": np.concatenate(order),
           "spans": np.concatenate(spans), "rows": np.concatenate(rows)}
    out = {name: np.ascontiguousarray(a, dtype=np.float64) for name, a in out.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[dump] {total / 1e6:.1f} MB of outputs -> {out_dir}")


def numa_cpus_of_gpu(index):
    """CPUs of the NUMA node the GPU hangs off (pinned buffers allocated by a thread bound there are node-local);
    None when the topology cannot be read."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return sorted(cpus) or None
    except Exception:
        return None


def config_block(n, R, label="4x32x8"):
    """The `config` both arms print (the reference arm runs a bounded sample of the same workload)."""
    return {"workload": f"{n}-job synthetic trace x {R} replicas/GPU (distinct seeds), {label} cluster, fifo+yarn",
            "jobs_per_replica": n, "replicas_per_gpu": R, "cluster": label, "policy": "fifo", "scheme": "yarn",
            "l2": "inputs + outputs of a step (GBs per GPU) exceed the 126 MB L2"}


POLICY_SETUP = {"sjf": dict(), "dlas": dict(num_queue=4, queue_limit=[3600, 7200, 18000]),
                "dlas-gpu": dict(num_queue=4, queue_limit=[3600, 7200, 18000])}


def make_policy(name, table):
    from gpuschedule_b200 import capi
    from gpuschedule_b200 import policies as gpol
    if name == "fifo":
        return capi.make_policy("fifo")
    if name == "gittins":
        return capi.make_policy("gittins", gittins_delta=3250.0,
                                gittins_table=gpol.build_gittins_table(gpol.gittins_samples(table), 3250.0))
    return capi.make_policy(name, **POLICY_SETUP[name])


def policy_measure(name, cluster, tabs, device, steps=1, check=True):
    """Event-driven policy kernels (BASELINE configs C2-C4 on one GPU): device-timed events/s over `tabs` replicas, the
    algorithmic bytes of SURVEY 8(d) -- per event (runnable jobs)*32 + M*16 + 64 -- from the rows of a sample of the
    replicas, one replica compared field by field with oracle/policy_oracle.c, which is also the timed CPU leg."""
    from gpuschedule_b200 import capi
    pols = [make_policy(name, t) for t in tabs]
    m = cluster.num_switch * cluster.num_node_p_switch
    with capi.Engine(device=device, nsims=len(tabs)) as pe:
        for i, t in enumerate(tabs):
            pe.config(i, cluster, pols[i])
            pe.load_trace_packed(i, t.packed())
        run_to_done(pe, 0)
        cap = max(pe.stats(i).ticks for i in range(len(tabs))) + 64
        ms = 0.0
        for _ in range(steps):
            pe.reset()
            run_to_done(pe, cap)
            ms += pe.stats(0).kernel_ms
        ms /= steps
        ev = sum(pe.stats(i).events for i in range(len(tabs)))
        sample = list(range(min(4, len(tabs))))
        alg = 0
        for i in sample:
            rows = pe.fetch_rows(i)
            alg += int((rows["running"].astype(np.int64) + rows["queued"]).sum()) * 32 + len(rows) * (m * 16 + 64)
        alg = alg / len(sample) * len(tabs)
        rows0, (recs0, order0), st0 = pe.fetch_rows(0), pe.fetch_jobs(0), pe.stats(0)
    out = {"value": ev / (ms / 1e3), "unit": UNIT, "ms": ms, "replicas": len(tabs), "jobs_per_replica": tabs[0].n,
           "kernel": "gs_dlas_warp_kernel" if name.startswith("dlas") else "gs_sortpol_warp_kernel"}
    peak, src = peaks()
    ach = alg / (ms / 1e3) / 1e9
    out["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                       "algorithmic_bytes_per_launch": alg, "peak_source": src,
                       "bytes_model": "SURVEY 8(d): per event (runnable jobs)*32 + M*16 + 64, summed over the events of a 4-replica sample, scaled"}
    if check:
        import oracle
        c0 = time.perf_counter()
        ref = oracle.run_policy(cluster, pols[0], tabs[0])
        t_cpu = time.perf_counter() - c0
        same = (rows0.tobytes() == ref.rows.tobytes() and recs0.tobytes() == ref.recs.tobytes()
                and np.array_equal(order0, ref.finish_order) and st0.events == ref.events)
        assert same, f"{name}: engine and oracle/policy_oracle.c disagree on replica 0"
        out["parity"] = "replica 0 == oracle/policy_oracle.c on every row, record and the finish order (asserted in this run)"
        out["cpu_baseline"] = {"value": ref.events / t_cpu, "unit": UNIT, "cores": 1, "kind": "port",
                               "sample": f"1 replica of {tabs[0].n} jobs, oracle/policy_oracle.c (restatement of the dead loop code, not reference code)"}
    return out


def ours(args):
    import torch
    import torch.distributed as dist
    from gpuschedule_b200 import capi
    from gpuschedule_b200 import log_manager as lm

    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"             # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    def barrier_sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from gpuschedule_b200 import dist as gdist
    red = gdist.Reducer(world, dev)

    if args.only_sharded:
        blk = sharded_block(args, rank, world, local, dev)
        if rank == 0:
            print(json.dumps(blk), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    cfg = apply_config(args)
    R, n = args.replicas, args.jobs
    cluster = capi.make_cluster(cfg["num_switch"], cfg["num_node_p_switch"], 8)
    M, G = cfg["num_switch"] * cfg["num_node_p_switch"], 8
    metric = cfg["metric"]
    if args.config != "c1":
        args.no_sharded = True                            # the C4 block and the CLI figure belong to the headline configuration
    t0 = time.time()
    seeds = gdist.replica_seeds(rank, world, R, base=BASE_SEED)
    if args.distinct and args.distinct < R:              # development only: fewer distinct traces, reused round robin
        seeds = [seeds[i % args.distinct] for i in range(R)]
    import concurrent.futures as cf
    with cf.ThreadPoolExecutor(min(32, len(os.sched_getaffinity(0)))) as ex:      # numpy releases the GIL in the generators
        made = dict(zip(sorted(set(seeds)), ex.map(lambda sd: fast_table(n, sd, rate=cfg["rate"]), sorted(set(seeds)))))
    tables = [made[sd] for sd in seeds]
    log(f"[rank {rank}] generated {len(made)} traces of {n} jobs in {time.time() - t0:.1f}s")

    if args.policy != "fifo":
        # secondary mode: one event-driven policy alone (device-timed value, roofline, oracle check of replica 0)
        out = policy_measure(args.policy, cluster, tables, local, steps=args.steps, check=(rank == 0))
        ev_all = red.sum(out["value"] * out["ms"] / 1e3)
        ms = red.max(out["ms"])
        if rank == 0:
            out.update({"metric": metric, "value": ev_all / (ms / 1e3), "n_gpus": world, "steps": args.steps,
                        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                        "vs_baseline": None, "data": "synthetic", "dtype": "int32/int64 (+f64 ranks)",
                        "config": {"workload": f"{n}-job synthetic trace x {R} replicas/GPU, 4x32x8, {args.policy}"}})
            print(json.dumps(out), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    if args.config != "c1":
        args.span_budget = 0.0                            # deep queues spread jobs over more nodes: keep the worst-case pool
    eng = capi.Engine(device=local, nsims=R)
    eng.set_span_budget(args.span_budget)
    for r in range(R):
        eng.config(r, cluster)
        eng.load_trace_packed(r, tables[r].packed())

    # ---- warm-up (also sizes the per-replica record windows so that one launch completes a run)
    totals = {}
    run_to_done(eng, 0, totals)                           # (a deep-queue run needs several default-sized windows)
    wins = [eng.window(r) for r in range(R)]
    ticks = [int(w.ticks) for w in wins]
    rows_cap = max(t[0] for t in totals.values()) + 256
    qrows_cap = max(t[1] for t in totals.values()) + 256
    eng.set_queue_rows_cap(qrows_cap)
    for _ in range(max(args.warmup - 1, 2)):
        eng.reset()
        run_to_done(eng, rows_cap)

    # ---- timed: K steps, traces resident in HBM; a step = reset + one full simulation of every replica
    sampler = ClockSampler(local)
    launches0 = eng.launch_count()
    barrier_sync()
    sampler.start()
    w0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        eng.reset()
        run_to_done(eng, rows_cap)
        dev_ms += eng.stats(0).kernel_ms
    barrier_sync()
    wall_ms = (time.perf_counter() - w0) * 1e3
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    st = [eng.stats(r) for r in range(R)]
    wins = [eng.window(r) for r in range(R)]
    events_rank = sum(s.events for s in st)
    ticks_rank = sum(s.ticks for s in st)
    evals_rank = sum(s.placement_evals for s in st)
    spans_rank = sum(int(w.spans_used) for w in wins)
    recs_rank = sum(int(w.ev_rows) + int(w.q_rows) for w in wins)      # (one window per run once the capacities are sized)
    dev_ms = red.max(dev_ms)
    wall_ms = red.max(wall_ms)
    events_all = red.sum(events_rank)
    value = events_all / (dev_ms / args.steps / 1e3)
    if args.dump_outputs and rank == 0:                   # rank 0's replicas are those of a one-GPU run
        dump_outputs(eng, args.dump_outputs)

    if args.value_only:
        if rank == 0:
            print(json.dumps({"value": value, "ms_per_step": dev_ms / args.steps, "replicas_per_gpu": R,
                              "records_per_tick": recs_rank / ticks_rank}), flush=True)
        eng.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- single replica (the headline configuration itself: ONE 100k-job simulation on one GPU)
    single = None
    if rank == 0:
        with capi.Engine(device=local, nsims=1) as e1:
            e1.config(0, cluster)
            e1.load_trace_packed(0, tables[0].packed())
            run_to_done(e1, 0)
            best = None
            for _ in range(3):
                e1.reset()
                run_to_done(e1, rows_cap)
                ms1 = e1.stats(0).kernel_ms
                best = ms1 if best is None else min(best, ms1)
            single = {"value": e1.stats(0).events / (best / 1e3), "unit": UNIT, "ms": best,
                      "note": "one %d-job simulation alone on the GPU: one warp, latency bound by construction" % n}

    # ---- roofline of the dominant kernel (gs_tick2_kernel), per launch, this rank's GPU.  Algorithmic bytes are
    # SURVEY 8(d)'s: job table in + job record out (56 B/job), one 16-B span per (job, node), one 64-B statistics
    # row per simulated tick -- the information the launch produces, whatever encoding the engine writes it in.
    alg_bytes = R * n * 56 + spans_rank * 16 + ticks_rank * 64
    written = R * n * (32 + 4 + 4) + spans_rank * 8 + recs_rank * 24
    peak, peak_src = peaks()
    ach = alg_bytes / (dev_ms / args.steps / 1e3) / 1e9
    traffic, traffic_src = None, None
    try:      # DRAM bytes per launch from the committed ncu --set full capture of THIS kernel at THIS replica count
        tj = json.load(open(os.path.join(REPO, "profiles", "r02_tick2_kernel_traffic.json")))
        if tj["jobs_per_replica"] == n:
            traffic = tj["dram_bytes_per_replica"] * R
            traffic_src = ("dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture at %d replicas "
                           "(profiles/r02_tick2_kernel_traffic.json)%s" % (tj["replicas"], "" if tj["replicas"] == R else ", scaled per replica to %d" % R))
    except Exception:
        traffic = None
    roofline = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": "gs_tick2_kernel", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "bytes_read_or_written_once_by_design": written,
                "records_per_tick": recs_rank / ticks_rank,
                "ticks_per_s": ticks_rank * world / (dev_ms / args.steps / 1e3),
                "candidate_evals_per_s": evals_rank * world / (dev_ms / args.steps / 1e3)}

    # ---- end to end through the C ABI with HOST buffers.  K host threads, each with its own engine handle (own
    # stream) over a slice of the replicas; every step each thread uploads its traces from page-locked host memory
    # (gs_load_trace_packed, asynchronous), runs them, and reads back every record of every replica into page-locked
    # host memory (gs_fetch_compact + gs_sync): statistics records, queue records, per-job results, finish order, spans.
    eng.close()                                          # free the HBM of the value run first
    K = max(1, min(args.e2e_threads, R))
    slices = [list(range(k, R, K)) for k in range(K)]
    e2e_steps = max(1, args.e2e_steps)
    results = [None] * K
    errors = []
    ready_evt = threading.Barrier(K + 1)                 # every thread has done its warm-up step
    start_evt = threading.Barrier(K + 1)
    end_evt = threading.Barrier(K + 1)                   # reached after the last timed step, BEFORE buffers are freed
    numa = numa_cpus_of_gpu(local)
    span_budget_e2e = (max(int(w.spans_used) for w in wins) + 64) / n
    stagger_unit = 0.25 + 0.6 * (dev_ms / args.steps / 1e3)       # rough length of a step's copy phases, seconds

    import ctypes as C
    numa = None if args.no_numa else numa

    class Half:
        """one engine handle over half of a thread's replicas, with its page-locked input block and output blocks"""

        def __init__(self, reps):
            self.reps = reps
            self.e = e = capi.Engine(device=local, nsims=len(reps))
            e.set_async(True)
            e.set_span_budget(span_budget_e2e)            # capacities sized by the warm-up run: the copied blocks carry little slack
            e.set_queue_rows_cap(qrows_cap)
            self.pin_in = capi.PinnedBuffer(len(reps) * n * 32)
            block = self.pin_in.view(capi.JOBIN_DTYPE, len(reps) * n)
            for i, r in enumerate(reps):
                block[i * n:(i + 1) * n] = tables[r].packed()      # the step's inputs live in host memory
                e.config(i, cluster)
            self.n_each = np.full(len(reps), n, dtype=np.int64)
            self.p_in, self.p_n = block.ctypes.data_as(C.c_void_p), self.n_each.ctypes.data_as(C.POINTER(C.c_int64))
            self.pin_out = self.out = self.lay = self.p_out = None
            self.pitch = 0
            self.pending = False                          # a read-back is in flight

        def load(self):                                   # ONE strided upload (asynchronous)
            if self.e.lib.gs_load_traces_packed(self.e.h, self.p_in, n * 32, self.p_n) != 0:
                raise capi.GsError("gs_load_traces_packed failed: " + self.e.lib.gs_last_error(self.e.h).decode())
            return len(self.reps) * n * 32

        def run(self):
            run_to_done(self.e, rows_cap)

        def fetch(self):                                  # ONE strided read-back (asynchronous)
            if self.pin_out is None:                      # first step: the result-block layout is known now
                self.lay = self.e.result_layout(0)
                self.pitch = (int(self.lay.block_bytes) + 255) // 256 * 256
                self.pin_out = capi.PinnedBuffer(len(self.reps) * self.pitch)
                self.out = self.pin_out.view(np.uint8, len(self.reps) * self.pitch)
                self.p_out = self.out.ctypes.data_as(C.c_void_p)
            if self.e.lib.gs_fetch_results(self.e.h, 0, len(self.reps), self.p_out, self.pitch) != 0:
                raise capi.GsError("gs_fetch_results failed: " + self.e.lib.gs_last_error(self.e.h).decode())
            self.pending = True

        def finish(self, win):
            """wait for the read-back and touch every replica's results -> (valid bytes, copied bytes, checksum, events)"""
            self.e.sync()
            self.pending = False
            valid = chk = ev = 0
            for i in range(len(self.reps)):
                self.e.lib.gs_window(self.e.h, i, C.byref(win))
                evb, qrb, neb, jb, od, sp = capi.Engine.result_views(self.out, self.pitch, i, self.lay, win)
                valid += 24 * (win.ev_rows + win.q_rows) + 8 * win.node_events + 4 * n + 4 * win.finished + int(self.lay.span_bytes) * win.spans_used
                chk += int(evb[-1]["finished"]) + int(jb[0]["start"]) + int(od[-1]) + int(sp[-1]["devmask"])
                ev += n + 2 * win.finished                # arrivals + starts + completions of a finished run
            return valid, len(self.reps) * int(self.lay.block_bytes), chk, ev

        def close(self):
            self.pin_in.free()
            if self.pin_out is not None:
                self.pin_out.free()
            self.e.close()

    def worker(k):
        try:
            if numa:
                os.sched_setaffinity(0, numa)            # this thread only: its pinned allocations are node-local
            mine = slices[k]
            # two handles per thread: while one half's results travel to the host, the other half uploads and simulates
            cut = (len(mine) + 1) // 2
            halves = [Half(mine[:cut])] + ([Half(mine[cut:])] if len(mine) > cut else [])
            ph = dict(load=0.0, run=0.0, finish=0.0)
            h2d = d2h = d2h_copied = chk = ev_cnt = 0
            win = capi.GsWindowInfo()
            for step in range(e2e_steps + 1):            # step 0 = untimed warm-up (allocations)
                if step == 1:
                    for hf in halves:                     # drain the warm-up step completely
                        if hf.pending:
                            hf.finish(win)
                    ready_evt.wait()                      # warm-up done everywhere; main synchronises the ranks ...
                    start_evt.wait()                      # ... and the timed region starts for all threads + main
                    ph = dict(load=0.0, run=0.0, finish=0.0)
                    h2d = d2h = d2h_copied = chk = ev_cnt = 0
                    if k % 2 == 1 and args.e2e_stagger > 0:
                        time.sleep(args.e2e_stagger * stagger_unit)     # odd threads run a fraction of a step behind the even ones
                for hf in halves:
                    other = halves[1 - halves.index(hf)] if len(halves) == 2 else None
                    c0 = time.perf_counter()
                    if hf.pending:                        # (single-handle case) its own previous read-back first
                        v, cp, ck, ev = hf.finish(win); d2h += v; d2h_copied += cp; chk += ck; ev_cnt += ev
                    h2d += hf.load()
                    c1 = time.perf_counter(); ph["load"] += c1 - c0
                    hf.run()                              # the other half's read-back proceeds on its own stream meanwhile
                    c2 = time.perf_counter(); ph["run"] += c2 - c1
                    hf.fetch()
                    if other is not None and other.pending:
                        v, cp, ck, ev = other.finish(win); d2h += v; d2h_copied += cp; chk += ck; ev_cnt += ev
                    ph["finish"] += time.perf_counter() - c2
            c2 = time.perf_counter()
            for hf in halves:                             # the last read-backs belong to the timed region
                if hf.pending:
                    v, cp, ck, ev = hf.finish(win); d2h += v; d2h_copied += cp; chk += ck; ev_cnt += ev
            ph["finish"] += time.perf_counter() - c2
            end_evt.wait()                                # the timed region ends when the slowest thread gets here
            # the records really are the run: decode one replica of this thread and compare with the value run
            hf = halves[0]
            hf.e.lib.gs_window(hf.e.h, 0, C.byref(win))
            evb, qrb, neb, jb, od, sp = capi.Engine.result_views(hf.out, hf.pitch, 0, hf.lay, win)
            rows = lm.expand_rows(evb, qrb, neb, win.row_first, win.ticks, M, G)
            assert len(rows) == ticks[mine[0]] and int(rows["finished"][-1]) == n and int(rows["now"][-1]) == ticks[mine[0]]
            results[k] = (ph, h2d // e2e_steps, d2h // e2e_steps, chk, ev_cnt // e2e_steps, d2h_copied // e2e_steps)
            for hf in halves:
                hf.close()
        except Exception as exc:                          # surface worker failures in the main thread
            errors.append(exc)
            for b_ in (ready_evt, start_evt, end_evt):
                try:
                    b_.abort()
                except Exception:
                    pass

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(K)]
    for t in threads:
        t.start()
    try:
        ready_evt.wait()
        barrier_sync()                                    # all ranks start their timed region together
        start_evt.wait()                                  # released together with the workers' timed steps
    except threading.BrokenBarrierError:
        pass
    w0 = time.perf_counter()
    try:
        end_evt.wait()                                    # every thread has finished (and synchronised) its last timed step
    except threading.BrokenBarrierError:
        pass
    e2e_wall = time.perf_counter() - w0
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    barrier_sync()
    e2e_ms = red.max(e2e_wall * 1e3) / e2e_steps
    h2d = sum(r[1] for r in results); d2h = sum(r[2] for r in results)
    checksum = sum(r[3] for r in results)
    assert sum(r[4] for r in results) == events_rank, "e2e run simulated a different number of events"
    ph = {k: max(r[0][k] for r in results) for k in ("load", "run", "finish")}
    d2h_copied = sum(r[5] for r in results)
    e2e = {"value": events_all / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": int(red.sum(h2d)), "d2h_bytes_per_step": int(red.sum(d2h_copied)),
           "d2h_valid_bytes_per_step": int(red.sum(d2h)),
           "steps": e2e_steps, "host_threads": K, "pinned_buffers_numa_local": bool(numa),
           "timing": "wall clock between barrier+synchronize around the timed steps of all threads, max over ranks",
           "phase_ms_per_step_slowest_thread": {k: v * 1e3 / e2e_steps for k, v in ph.items()},
           "pipeline": "two engine handles per host thread: the strided read-back of one half overlaps the strided upload and the kernel of the other",
           "result_format": "compact records (24-byte gs_evrow / gs_qrow, gs_nodeev, start ticks, finish order, 8-byte gs_cspan), one strided copy per handle each way "
                            "(d2h_bytes counts the copied blocks incl. their unused capacity); one replica per thread is decoded to full rows and checked",
           "checksum": checksum}

    if args.e2e_only:
        probe = {}
        try:                                              # what one stream gets out of the link, for orientation
            hbuf = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
            dbuf = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
            for name, (dst, src) in (("d2h", (hbuf, dbuf)), ("h2d", (dbuf, hbuf))):
                dst.copy_(src, non_blocking=True); torch.cuda.synchronize()
                t0 = time.perf_counter(); dst.copy_(src, non_blocking=True); torch.cuda.synchronize()
                probe[name + "_gbs_1GiB_one_stream"] = (1 << 30) / (time.perf_counter() - t0) / 1e9
        except Exception as exc:
            probe["error"] = repr(exc)
        if rank == 0:
            print(json.dumps({"e2e": e2e, "copy_probe": probe, "value": value, "replicas_per_gpu": R}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- secondary measurements (rank 0, N=1): the event-driven policies of BASELINE configs C2-C4 on the same
    # cluster (device-timed, 1 warm-up + 1 timed run each, replica 0 checked against the oracle) and the stateless scoring kernel
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        extras = {}
        rp = min(R, args.policy_replicas)
        pn = min(n, 100000)                              # C2: 10k-job sjf; C3 / C4: 100k jobs (c5: the same sizes on 16x64x8)
        for name, njobs in (("sjf", min(pn, 10000)), ("dlas-gpu", pn), ("gittins", pn)):
            tabs = tables[:rp] if njobs == n else [fast_table(njobs, sd, rate=cfg["rate"]) for sd in gdist.replica_seeds(0, 1, rp, base=BASE_SEED)]
            try:
                extras[name] = policy_measure(name, cluster, tabs, local)
            except Exception as exc:                      # a secondary line never costs the main one
                extras[name] = {"error": repr(exc)}
        try:
            import contextlib
            import io
            buf = io.StringIO()
            pa = argparse.Namespace(place_jobs=16 * 1024 * 1024, warmup=2, steps=3)
            with contextlib.redirect_stdout(buf):
                place_mode(pa)
            pj = json.loads(buf.getvalue().strip().splitlines()[-1])
            extras["place_batch"] = {"value": pj["value"], "unit": pj["unit"], "kernel_ms": pj["kernel_ms"], "jobs": pj["jobs"],
                                     "candidate_evals_per_s": pj["candidate_evals_per_s"], "roofline_frac": pj["roofline"]["frac"],
                                     "achieved_gbs": pj["roofline"]["achieved"]}
        except Exception as exc:
            extras["place_batch"] = {"error": str(exc)}
        # row f3: the command line end to end on the headline trace (ingest, engine, RNG-column replay, CSV writing)
        try:
            if args.config != "c1":
                raise RuntimeError("measured on the headline configuration only")
            import glob
            import shutil
            import tempfile
            from gpuschedule_b200 import tracegen
            tmp = tempfile.mkdtemp(prefix="gs_cli_")
            tracegen.write_trace(os.path.join(tmp, "t.csv"), n, seed=BASE_SEED, rate=0.5)
            cmd = [sys.executable, os.path.join(REPO, "run_sim.py"), "--num_switch", "4", "--num_node_p_switch", "32", "--num_gpu_p_node", "8",
                   "--scheme", "yarn", "--schedule", "fifo", "--trace_file", "t.csv", "--log_path", "cli", "--seed", "7"]
            best, runs_s = None, []
            for _ in range(3):                              # run 1 parses the trace with pandas and leaves the parsed table under log/.trace_cache
                c0 = time.perf_counter()
                cp = subprocess.run(cmd, cwd=tmp, capture_output=True, text=True, timeout=120)
                dt = time.perf_counter() - c0
                runs_s.append(dt)
                best = dt if best is None else min(best, dt)
            runs = sorted(glob.glob(os.path.join(tmp, "log", "cli", "*")))
            lines = sum(1 for _ in open(os.path.join(runs[-1], "cluster.csv"))) - 1
            jl = sum(1 for _ in open(os.path.join(runs[-1], "job.csv"))) - 1
            extras["cli"] = {"seconds": best, "cmd": "python run_sim.py --scheme yarn --schedule fifo (4x32x8) on the %d-job trace, --seed 7" % n,
                             "seconds_first_run": runs_s[0], "runs_s": runs_s,
                             "cluster_csv_rows": lines, "job_csv_rows": jl, "events_per_s": 3.0 * jl / best, "rc": cp.returncode,
                             "note": "process start to exit: imports, CUDA context, trace ingest, engine, host replay of the sampled "
                                     "utilisation column (numpy's sequential legacy generator), CSV formatting.  seconds_first_run parses "
                                     "the trace with pandas (whose import alone is ~1 s); the later runs -- a sweep replays one trace "
                                     "many times -- read the parsed table from --trace_cache.  Round 1: 11.4 s"}
            shutil.rmtree(tmp, ignore_errors=True)
        except Exception as exc:
            extras["cli"] = {"error": repr(exc)}
        # widening row f1 (horus / gandiva / horus+ engine): its own process with a time limit, so that nothing it
        # does can cost the main measurement
        try:
            hp = subprocess.run([sys.executable, os.path.abspath(__file__), "--mode", "horus", "--horus-replicas", "9472"],
                                capture_output=True, text=True, timeout=400)
            line = [ln for ln in hp.stdout.splitlines() if ln.startswith("{")]
            extras["horus"] = json.loads(line[-1]) if line else {"error": (hp.stderr or "no output")[-400:]}
        except Exception as exc:
            extras["horus"] = {"error": repr(exc)}

    # ---- CPU baseline: the oracle port, 1 thread, bounded sample (rank 0, N=1 only)
    cpu = None
    cpu_tight = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        t_cpu, ev_cpu, k = 0.0, 0, 0
        if args.config == "c1":
            while t_cpu < args.cpu_seconds and k < R:
                c0 = time.perf_counter()
                ref = oracle.run_fifo(cluster, tables[k], rows_cap=max(ticks) + 128, want_spans=False)
                t_cpu += time.perf_counter() - c0
                ev_cpu += ref.events
                assert ref.ticks == ticks[k] and ref.events == st[k].events, "engine/oracle disagree"
                k += 1
            sample = f"{k} replica(s) of the {n}-job trace, full runs, oracle/gsched_oracle.c single thread"
        else:       # the literal port re-scans M x G devices per tick: a full 1M-job run takes ~20 minutes, so a bounded sample
            small = fast_table(20000, BASE_SEED, rate=cfg["rate"])
            c0 = time.perf_counter()
            ref = oracle.run_fifo(cluster, small, want_spans=False)
            t_cpu, ev_cpu, k = time.perf_counter() - c0, ref.events, 1
            sample = f"one 20000-job trace of the same generator and cluster (bounded sample), oracle/gsched_oracle.c single thread"
        cpu = {"value": ev_cpu / t_cpu, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample, "host_cores": os.cpu_count()}
        cpu_tight = tight_yardstick(cluster, tables[:1], 1, ticks[0])
        try:                                                # and on every host core (memory bound long before 128 threads)
            ncores = len(os.sched_getaffinity(0))
            cpu_tight["all_cores"] = tight_yardstick(cluster, tables[:ncores], min(ncores, len(tables)))
        except Exception as exc:                            # noqa: BLE001
            cpu_tight["all_cores"] = {"error": repr(exc)}

    sharded = None
    if not args.no_sharded:
        try:
            sharded = sharded_block(args, rank, world, local, dev)
        except Exception as exc:                          # the secondary block never costs the main line
            sharded = {"error": repr(exc)}

    if rank == 0:
        out = {
            "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32/int64 (+f64 durations)",
            "data": "synthetic",
            "config": config_block(n, R, cfg["label"]),
            "run": {"parallelism": f"replicas x{world} GPUs, no data-path collective", "events_per_step": events_all,
                    "ticks_per_step": red_ticks_all(ticks_rank, world), "step_bytes_per_gpu": written},
            "wall_ms_per_step": wall_ms / args.steps,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "single_replica": single,
            "roofline": roofline, "cpu_baseline": cpu, "cpu_tight": cpu_tight,
            "vs_cpu_tight_one_core": (None if not cpu_tight else {"device_timed": value / cpu_tight["value"], "e2e": e2e["value"] / cpu_tight["value"],
                                                                   "single_replica": single["value"] / cpu_tight["value"]}),
            "vs_cpu_tight_all_cores": (None if not cpu_tight or "value" not in cpu_tight.get("all_cores", {}) else
                                       {"device_timed": value / cpu_tight["all_cores"]["value"], "e2e": e2e["value"] / cpu_tight["all_cores"]["value"],
                                        "cores": cpu_tight["all_cores"]["cores"]}),
            "sharded": sharded, "secondary": extras,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def sharded_block(args, rank, world, local, dev):
    """BASELINE config C4: ONE gittins simulation, on one GPU and sharded over the `world` GPUs of the box (rank
    evaluation split by chunks of the runnable list, one NVLink peer-store exchange per event inside the persistent
    kernel; include/gsched.h gs_comm_*).  Every rank runs both and compares the bytes.  Two traces: the BASELINE one
    (100k jobs, 0.5 arrivals per tick: ~20 runnable jobs, one chunk -- nothing to split, the exchange is pure cost) and an
    overloaded one (12k jobs at 20 per tick: a runnable list of several thousand)."""
    from gpuschedule_b200 import capi
    from gpuschedule_b200 import dist as gdist
    cluster = capi.make_cluster(4, 32, 8)
    red = gdist.Reducer(world, dev)

    # Every rank reaches the same collectives (barriers, reductions, the handle all-gather) whatever fails locally: a
    # failure is carried as `err` and agreed on afterwards, so a rank with a problem cannot leave its peers in a collective.
    def timed(eng, table, pol, reps=2, err=None):
        best, events, blob, cap = None, 0, None, 0
        if err is None:
            try:
                eng.config(0, cluster, pol)
                eng.load_trace_packed(0, table.packed())
                run_to_done(eng, 0)                      # (sharded: a peer that never starts ends this with GS_ERR_COMM after ~5 s)
                cap = eng.stats(0).ticks + 64
            except Exception as exc:                      # noqa: BLE001
                err = repr(exc)
        for _ in range(reps):
            red.barrier()
            if err is None:
                try:
                    eng.reset()
                    run_to_done(eng, cap)
                    ms = eng.stats(0).kernel_ms
                    best = ms if best is None else min(best, ms)
                except Exception as exc:                  # noqa: BLE001
                    err = repr(exc)
        if err is None:
            try:
                rows = eng.fetch_rows(0)
                recs, order = eng.fetch_jobs(0)
                events, blob = eng.stats(0).events, (rows.tobytes(), recs.tobytes(), order.tobytes())
            except Exception as exc:                      # noqa: BLE001
                err = repr(exc)
        return best, events, blob, err

    def one(n, rate, reps=2):
        table = fast_table(n, BASE_SEED, rate=rate)
        pol = make_policy("gittins", table)
        with capi.Engine(device=local, nsims=1) as e1:
            ms1, events, single, err1 = timed(e1, table, pol, reps)
        if red.sum(1.0 if err1 else 0.0) > 0:
            return {"jobs": n, "arrivals_per_tick": rate, "error": err1 or "another rank failed its single-GPU run"}
        ms1 = red.max(ms1)
        out = {"jobs": n, "arrivals_per_tick": rate, "events": int(events),
               "single_gpu": {"ms": ms1, "events_per_s": events / (ms1 / 1e3)}}
        if world > 1:
            # "always": an exchange on every event (what the north-star sketches); "above_256": events whose runnable list
            # is at most 256 jobs long are evaluated by every rank itself, without sending anything; "sharded": the library's
            # default after gs_comm_init, which exchanges only when the caller sets a threshold (no measured list pays for one)
            for key, min_rn in (("sharded_always_exchange", 0), ("sharded_above_256", 256), ("sharded", None)):
                with capi.Engine(device=local, nsims=1) as e2:
                    err, hnd = None, bytes(64)
                    try:
                        hnd = e2.comm_prepare(n)
                    except Exception as exc:              # noqa: BLE001
                        err = repr(exc)
                    handles = gdist.exchange_comm_handles(hnd, world, dev)
                    if err is None:
                        try:
                            e2.comm_init(rank, handles)
                            if min_rn is not None:
                                e2.comm_set_min_runnable(min_rn)
                        except Exception as exc:          # noqa: BLE001
                            err = repr(exc)
                    msN, eventsN, shard, err = timed(e2, table, pol, reps, err)
                    exchanges, us = (0, 0.0)
                    if err is None:
                        exchanges, us = e2.comm_stats()
                if red.sum(1.0 if err else 0.0) > 0:
                    out[key] = {"error": err or "another rank failed"}
                    continue
                same = red.sum(1.0 if (shard == single and eventsN == events) else 0.0)
                msN = red.max(msN)
                out[key] = {"ms": msN, "events_per_s": events / (msN / 1e3), "min_runnable_for_exchange": min_rn if min_rn is not None else "library default (never)", "exchanges": exchanges,
                            "exchange_us_mean": red.max(us), "ranks_identical_to_single_gpu": int(same), "speedup_vs_single_gpu": ms1 / msN}
        return out

    blk = {"policy": "gittins", "n_gpus": world,
           "exchange": "NVLink peer stores + flag words inside the persistent kernel (no NCCL call on the data path)",
           "baseline_trace": one(args.sharded_jobs, args.sharded_rate)}
    if not args.sharded_skip_overloaded:
        blk["overloaded_trace"] = one(12000, 20.0, reps=1)
    return blk


def red_ticks_all(ticks_rank, world):
    return ticks_rank * world            # every rank simulates the same number of replicas of statistically equal traces


def tight_yardstick(cluster, tables, threads, expect_ticks=None, seconds=3.0):
    """oracle/tight2_cpu.c -- the GPU engine's own event-stepped algorithm as tight single-thread C -- on `threads`
    host threads, one replica each (ctypes releases the GIL): the strongest CPU competitor we could write."""
    import concurrent.futures as cf
    import oracle
    runners = [oracle.Tight2(cluster, t) for t in tables[:threads]]
    with cf.ThreadPoolExecutor(threads) as ex:
        first = list(ex.map(lambda r: r.run(), runners))
        if expect_ticks is not None:
            assert first[0][0] == expect_ticks
        t0 = time.perf_counter(); ev_t = 0; reps = 0
        while time.perf_counter() - t0 < seconds:
            ev_t += sum(e for _, e in ex.map(lambda r: r.run(), runners)); reps += 1
        dt = time.perf_counter() - t0
    return {"value": ev_t / dt, "unit": UNIT, "cores": threads,
            "kind": "tight C restatement of the ENGINE's event-stepped algorithm (oracle/tight2_cpu.c), not reference code; "
                    "writes the same compact records",
            "sample": f"{reps} rounds of {threads} replica(s) of the {tables[0].n}-job trace, one per thread"}


def place_mode(args):
    """Secondary measurement: gs_place_batch, the stateless (job x candidate node) scoring kernel.
    b job requests against one 128-node cluster state; kernel-only time from the library's CUDA
    events; algorithmic bytes = 16 B request in + 8 B (first node, nodes used) out per job."""
    from gpuschedule_b200 import capi
    rng = np.random.default_rng(5)
    m, g = 128, 8
    cluster = capi.make_cluster(4, 32, g)
    nodes = np.zeros(m, dtype=capi.NODE_DTYPE)
    for i in range(m):
        k = int(rng.integers(0, g + 1))
        nodes["busy_mask"][i] = sum(1 << int(d) for d in rng.choice(g, size=k, replace=False))
        nodes["cpu_used"][i] = 12 * k
        nodes["mem_used"][i] = 60 * k
    b = args.place_jobs
    jobs = np.zeros(b, dtype=capi.JOBREQ_DTYPE)
    jobs["gpu_per_task"] = 1
    jobs["gpus"] = rng.choice([1, 2, 4, 8, 16, 32], size=b, p=[.35, .2, .2, .15, .07, .03])
    jobs["mem_bytes"] = rng.integers(512, 16384, size=b).astype(np.int64) << 20
    with capi.Engine(device=0, nsims=1) as eng:
        best = None
        for _ in range(args.warmup + args.steps):
            first, used, _, ms = eng.place_batch(cluster, nodes, jobs)
            best = ms if best is None else min(best, ms)
        placed = int((first >= 0).sum())
    peak, src = peaks()
    gbs = b * 24 / (best / 1e3) / 1e9
    print(json.dumps({"metric": "gs_place_batch jobs scored/s (128-node cluster state)", "value": b / (best / 1e3),
                      "unit": "jobs/s", "kernel_ms": best, "jobs": b, "placeable": placed,
                      "candidate_evals_per_s": b * m / (best / 1e3),
                      "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                                   "algorithmic_bytes_per_launch": b * 24, "peak_source": src,
                                   "kernel": "gs_place_kernel", "traffic": None}}), flush=True)


def horus_mode(args):
    """Secondary measurement (widening row f1): the utilisation-aware engine, `--horus-replicas` independent
    horus simulations (one thread each, gs_horus_kernel) of `--horus-jobs`-job traces on a 2x4x8 cluster.
    Replicas have distinct traces and read one common numpy stream (seed 0).  value = events / kernel time
    (library CUDA events); cpu_baseline = oracle/horus_oracle.c on one host core over a sample of replicas."""
    import oracle
    from gpuschedule_b200 import capi
    R, n = args.horus_replicas, args.horus_jobs
    cluster = capi.make_cluster(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8)
    tables = [fast_table(n, BASE_SEED + 1000 + r, rate=1.0) for r in range(R)]
    np.random.seed(0)
    stream = np.random.standard_normal(args.horus_stream)          # one numpy stream, shared by all replicas
    hp = capi.make_horus_params("horus", "horus", 5)
    with capi.HorusEngine(device=0, nsims=R) as eng:
        for r in range(R):
            eng.config(r, cluster, hp)
            eng.load_trace(r, tables[r])
        by_lanes = {}
        for lanes in ((32, 1) if args.horus_both_mappings else (1,)):   # 1 simulation per warp won round 1 (2.8x)
            eng.set_lanes(lanes)
            eng.load_stream(-1, stream)                    # (re)loading the stream starts the replicas over
            eng.run(rows_cap=args.horus_rows)
            by_lanes[lanes] = float(eng.stats(0).kernel_ms)
        st = [eng.stats(r) for r in range(R)]
        ms = min(by_lanes.values())
        events = sum(int(x.events) for x in st)
        ticks = sum(int(x.ticks) for x in st)
        draws = sum(int(x.draws) for x in st)
        assert all(x.done for x in st)
        rows0, util0, flags0, recs0, order0 = eng.fetch(0)
    ref = oracle.run_horus(cluster, tables[0], scheme="horus", schedule="horus", num_buffer=5, seed=0)
    assert rows0.tobytes() == ref.rows.tobytes() and util0.tobytes() == ref.util.tobytes(), "replica 0 differs from the oracle"
    if args.horus_scalar_only:                              # development: the scalar mapping's time alone
        print(json.dumps({"value": events / (ms / 1e3), "kernel_ms_by_lanes_per_warp": by_lanes, "replicas": R}), flush=True)
        return
    # horus+ (credit queues + k-means, raw word stream): a few replicas against the oracle, replica by replica
    plus = None
    try:
        k = 6
        np.random.seed(1)
        words = np.random.randint(0, 2 ** 32, size=args.horus_words, dtype=np.uint32)
        pp = capi.make_horus_params("horus+", "horus+", 15, 3)
        with capi.HorusEngine(device=0, nsims=k) as eng:
            for r in range(k):
                eng.config(r, cluster, pp)
                eng.load_trace(r, tables[r])
            eng.load_words(-1, words)
            eng.run(rows_cap=args.horus_rows)
            plus_ms = float(eng.stats(0).kernel_ms)
            same = 0
            for r in range(k):
                prow, putil, pflag, precs, porder = eng.fetch(r)
                pref = oracle.run_horus(cluster, tables[r], scheme="horus+", schedule="horus+", num_buffer=15, num_queue=3, seed=1)
                same += int(prow.tobytes() == pref.rows.tobytes() and putil.tobytes() == pref.util.tobytes()
                            and precs.tobytes() == pref.recs.tobytes() and np.array_equal(porder, pref.finish_order))
        plus = {"replicas": k, "identical_to_oracle": same, "kernel_ms": plus_ms}
    except Exception as exc:                                # noqa: BLE001 - reported, never fatal for the horus line
        plus = {"error": repr(exc)}
    sample = min(R, 64)
    t0 = time.perf_counter()
    cpu_ev = sum(oracle.run_horus(cluster, tables[r], scheme="horus", schedule="horus", num_buffer=5, seed=0).events for r in range(sample))
    cpu_s = time.perf_counter() - t0
    # the honest CPU yardstick: the ENGINE's own core (gs_horus_core.cuh, with its shortcuts) compiled for the host by the
    # test harness (tests/emu), one core, same replicas and stream -- what `cpu_tight` is for the fifo engine
    tight = None
    try:
        import tempfile
        sys.path.insert(0, os.path.join(REPO, "tests"))
        import emu
        with tempfile.TemporaryDirectory(prefix="gs_emu_") as tmp:
            emu.lib(os.path.join(tmp, "libhorus_emu.so"))       # loaded: the file may go with the directory
        k = min(R, 256)
        t0 = time.perf_counter()
        tight_ev = sum(emu.run_horus(cluster, hp, tables[r], stream, args.horus_rows)[6] for r in range(k))
        tight_s = time.perf_counter() - t0
        tight = {"value": tight_ev / tight_s, "unit": UNIT, "cores": 1,
                 "kind": "the engine's own core (gs_horus_core.cuh) built for the host with g++ -O2 (tests/emu), not reference code",
                 "sample": f"{k} of the {R} replicas, one thread",
                 "gpu_in_cores_of_it": (events / (ms / 1e3)) / (tight_ev / tight_s)}
    except Exception as exc:                                # noqa: BLE001
        tight = {"error": repr(exc)}
    # the warp-cooperative mapping (one simulation per warp, all lanes score together): LAST, in its own handle, so
    # that whatever it does cannot touch the numbers above
    coop = None
    try:
        with capi.HorusEngine(device=0, nsims=R) as eng:
            eng.set_lanes(0)
            for r in range(R):
                eng.config(r, cluster, hp)
                eng.load_trace(r, tables[r])
            eng.load_stream(-1, stream)
            eng.run(rows_cap=args.horus_rows)
            cst = [eng.stats(r) for r in range(R)]
            crow, cutil, cflag, crecs, corder = eng.fetch(0)
            coop = {"kernel_ms": float(cst[0].kernel_ms), "events": sum(int(x.events) for x in cst),
                    "events_per_s": sum(int(x.events) for x in cst) / (float(cst[0].kernel_ms) / 1e3),
                    "replica0_identical_to_oracle": bool(crow.tobytes() == ref.rows.tobytes() and cutil.tobytes() == ref.util.tobytes()
                                                         and crecs.tobytes() == ref.recs.tobytes()),
                    "same_event_total_as_scalar_mapping": sum(int(x.events) for x in cst) == events}
    except Exception as exc:                                # noqa: BLE001
        coop = {"error": repr(exc)}
    if isinstance(plus, dict) and "error" not in plus and "error" not in coop:
        try:                                                # horus+ under the cooperative mapping (indexed word stream)
            k = plus["replicas"]
            with capi.HorusEngine(device=0, nsims=k) as eng:
                eng.set_lanes(0)
                for r in range(k):
                    eng.config(r, cluster, pp)
                    eng.load_trace(r, tables[r])
                eng.load_words(-1, words)
                eng.run(rows_cap=args.horus_rows)
                same = 0
                for r in range(k):
                    prow, putil, pflag, precs, porder = eng.fetch(r)
                    pref = oracle.run_horus(cluster, tables[r], scheme="horus+", schedule="horus+", num_buffer=15, num_queue=3, seed=1)
                    same += int(prow.tobytes() == pref.rows.tobytes() and putil.tobytes() == pref.util.tobytes() and precs.tobytes() == pref.recs.tobytes())
                coop["horus_plus"] = {"replicas": k, "identical_to_oracle": same, "kernel_ms": float(eng.stats(0).kernel_ms)}
        except Exception as exc:                            # noqa: BLE001
            coop["horus_plus"] = {"error": repr(exc)}
    print(json.dumps({"metric": "horus simulated events/s (replica batch)", "value": events / (ms / 1e3), "unit": UNIT,
                      "kernel_ms": ms, "replicas": R, "jobs_per_replica": n, "ticks": ticks, "samples_drawn": draws,
                      "samples_per_s": draws / (ms / 1e3), "kernel": "gs_horus_kernel (one simulation per thread)", "kernel_ms_by_lanes_per_warp": by_lanes,
                      "parity": "replica 0 == oracle/horus_oracle.c == reference (tests/golden/horus_*)",
                      "horus_plus_device_check": plus, "cooperative_warp_mapping": coop,
                      "cpu_baseline": {"value": cpu_ev / cpu_s, "unit": UNIT, "cores": 1, "kind": "port",
                                       "sample": f"{sample} of the {R} replicas, oracle/horus_oracle.c, one thread"},
                      "cpu_tight": tight}), flush=True)


def reference(args):
    """The reference arm: the CPU port of the reference's loop (oracle/gsched_oracle.c) on ALL the host cores this
    process may use, one replica per thread.  The Python reference itself (186 events/s at N=10k, O(N^2)) cannot travel
    to the GPU box and could not finish one 100k-job replica in the time of the whole bench."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import concurrent.futures as cf
    import oracle
    from gpuschedule_b200 import capi
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cfg = apply_config(args)
    n = args.jobs
    cluster = capi.make_cluster(cfg["num_switch"], cfg["num_node_p_switch"], 8)
    oracle.lib()
    threads = max(1, min(cores, args.cpu_threads or cores))     # default: every core, always (same denominator in every record)
    n_run = n if args.config == "c1" else 20000                 # c5: bounded sample (the literal port needs ~20 min per 1M-job run)
    tables = [fast_table(n_run, BASE_SEED + r, rate=cfg["rate"]) for r in range(threads)]
    caps = [int(t.arrive_tick[-1]) + 2 * int(np.ceil(t.duration.max())) + 4096 for t in tables]

    def one(it):
        t, cap = it
        return oracle.run_fifo(cluster, t, rows_cap=cap, want_spans=False).events   # ctypes releases the GIL

    with cf.ThreadPoolExecutor(threads) as ex:
        work = list(zip(tables, caps))
        for _ in range(max(1, min(args.warmup, 2))):
            list(ex.map(one, work))
        t0 = time.perf_counter()
        events = 0
        for _ in range(args.steps):
            events += sum(ex.map(one, work))
        dt = time.perf_counter() - t0
    value = events / dt
    tight = tight_yardstick(cluster, tables, threads)
    sample = f"{threads} replicas of the {n_run}-job trace per step (one per thread on {cores} usable cores), full runs"
    out = {"impl": "reference", "metric": cfg["metric"], "value": value, "unit": UNIT,
           "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "int32/int64 (+f64 durations)", "data": "synthetic",
           "config": config_block(n, args.replicas, cfg["label"]),
           "run": {"replicas_per_step": threads, "host_threads": threads, "usable_cores": cores},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                            "note": "oracle/gsched_oracle.c: C restatement of the reference's Python loop "
                                    "(the Python reference itself: 186 events/s at N=10k, BASELINE.md)"},
           "cpu_tight": tight,
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c1", choices=sorted(CONFIGS), help="c1 = the BASELINE metric's configuration; c5 = 16x64x8, 1M-job traces")
    ap.add_argument("--jobs", type=int, default=None, help="jobs per trace (default: the configuration's)")
    ap.add_argument("--replicas", type=int, default=None, help="replicas per GPU, one warp each (default c1: 4144 = 148 SMs x 28 resident warps)")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--e2e-threads", type=int, default=16, help="host threads (one engine handle each) in the e2e run")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--value-only", action="store_true", help="kernel experiments: print the device-timed value and stop")
    ap.add_argument("--e2e-only", action="store_true", help="development: print the end-to-end block (with a copy-bandwidth probe) and stop")
    ap.add_argument("--e2e-stagger", type=float, default=0.5, help="fraction of a step by which every second host thread starts late, so that uploads, kernels and read-backs of different threads overlap")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the e2e threads to the GPU's NUMA node")
    ap.add_argument("--distinct", type=int, default=0, help="development: number of distinct traces (0 = one per replica)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary policy / place_batch measurements")
    ap.add_argument("--policy-replicas", type=int, default=2960, help="replicas of the secondary policy runs; 148 SMs x the 20 warps the policy kernels keep resident per SM")
    ap.add_argument("--no-sharded", action="store_true", help="skip the one-simulation-on-N-GPUs block (config C4)")
    ap.add_argument("--sharded-jobs", type=int, default=100000)
    ap.add_argument("--sharded-rate", type=float, default=0.5, help="arrivals per tick of the C4 trace (0.5 = the BASELINE generator; higher rates build a long runnable list)")
    ap.add_argument("--only-sharded", action="store_true", help="print the C4 block alone (development)")
    ap.add_argument("--sharded-skip-overloaded", action="store_true")
    ap.add_argument("--span-budget", type=float, default=1.5,
                    help="span-pool records per job (0 = worst case); the trace uses ~1.13, overflow is reported, never written")
    ap.add_argument("--policy", default="fifo", choices=["fifo", "sjf", "dlas", "dlas-gpu", "gittins"],
                    help="fifo = the headline (pinned) workload; others = secondary, event-driven policy kernel")
    ap.add_argument("--mode", default="sim", choices=["sim", "place", "horus"], help="place = gs_place_batch micro-benchmark; horus = utilisation-aware engine")
    ap.add_argument("--horus-replicas", type=int, default=2368)
    ap.add_argument("--horus-jobs", type=int, default=60)
    ap.add_argument("--horus-stream", type=int, default=4000000, help="standard-normal samples loaded per replica")
    ap.add_argument("--horus-rows", type=int, default=8192)
    ap.add_argument("--horus-both-mappings", action="store_true", help="also time 32 simulations per warp")
    ap.add_argument("--horus-scalar-only", action="store_true", help="development: time the scalar mapping and stop")
    ap.add_argument("--horus-words", type=int, default=6 << 20, help="raw generator words for the horus+ device check")
    ap.add_argument("--place-jobs", type=int, default=64 * 1024 * 1024)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "sim" or args.impl != "ours" or args.policy != "fifo" or args.only_sharded):
        ap.error("--dump-outputs writes the outputs of the fifo replica run (the default mode)")
    if args.mode == "place":
        place_mode(args)
    elif args.mode == "horus":
        horus_mode(args)
    elif args.impl == "reference":
        reference(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
