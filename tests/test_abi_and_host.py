"""CPU-side checks: the C-ABI library exports what include/gsched.h declares, fails
loudly without a GPU, and the host logic (flags, ingest, formatting) behaves."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import REPO


def _declared_symbols():
    names = set()
    for header in ("gsched.h", "gsched_horus.h"):
        src = open(os.path.join(REPO, "include", header)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"\b(gs_[a-z_0-9]+)\s*\(", src))
    return sorted(names)


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from gpuschedule_b200 import capi
    lib = ctypes.CDLL(capi.LIB_PATH)
    names = _declared_symbols()
    assert "gs_run" in names and "gs_place_batch" in names and "gs_horus_run" in names and len(names) >= 22
    for name in names:
        assert hasattr(lib, name), name
    assert lib.gs_abi_version() == 4


def test_library_is_built_for_sm_100a():
    from gpuschedule_b200 import _build, capi
    cuobjdump = os.path.join(os.path.dirname(_build.nvcc_path()), "cuobjdump")     # the toolkit need not be on PATH
    out = subprocess.run([cuobjdump, "-lelf", capi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback(have_gpu):
    if have_gpu:
        pytest.skip("GPU present")
    from gpuschedule_b200 import capi
    with pytest.raises(capi.GsError, match="no usable CUDA device|CUDA"):
        capi.Engine(device=0, nsims=1)


def test_product_never_imports_oracle():
    pkg = os.path.join(REPO, "gpuschedule_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h")):
                text = open(os.path.join(root, f)).read()
                assert "import oracle" not in text and "liboracle" not in text, f
    for f in ("run_sim.py", "execute.py"):
        p = os.path.join(REPO, f)
        if os.path.exists(p):
            assert "oracle" not in open(p).read(), f


def test_struct_sizes_match_header():
    from gpuschedule_b200 import capi, log_manager
    assert ctypes.sizeof(capi.GsCluster) == 56
    assert ctypes.sizeof(capi.GsRunStats) == 72
    assert log_manager.ROW_DTYPE.itemsize == 64
    assert log_manager.JOB_DTYPE.itemsize == 24
    assert capi.NODE_DTYPE.itemsize == 16 and capi.JOBREQ_DTYPE.itemsize == 16


def test_tracegen_is_deterministic_and_in_schema():
    from gpuschedule_b200 import ingest, tracegen
    a = tracegen.synth_columns(500, seed=3)
    b = tracegen.synth_columns(500, seed=3)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    for k in ingest.REQUIRED:
        assert k in a
    t = ingest.table_from_columns(a)
    assert t.n == 500 and np.all(np.diff(t.arrive_tick) >= 0)
    assert np.all(t.gpus % t.gpu_per_task == 0)


def test_ingest_filters_sorts_and_validates(tmp_path):
    import pandas as pd
    from gpuschedule_b200 import ingest, tracegen
    df = tracegen.synth_frame(30, seed=9)
    df.loc[3, "type"] = "interactive"
    df.loc[5, "minutes"] = np.nan
    p = tmp_path / "t.csv"
    df.sample(frac=1.0, random_state=1).to_csv(p, index=False)
    t = ingest.JobTraceReader(str(p)).prepare_jobs().table()
    assert t.n == 28 and len(set(t.label)) == 28
    assert t.arrive_tick[0] == 0 and np.all(np.diff(t.arrive_tick) >= 0)
    bad = tracegen.synth_frame(5, seed=1)
    bad.loc[2, "used_gpus"] = 0
    with pytest.raises(ValueError):
        ingest.table_from_frame(bad.assign(normalized_time=bad["normalized_time"] / 10000))
    with pytest.raises(SystemExit):
        ingest.JobTraceReader(str(tmp_path / "missing.csv"))


def test_flags_surface():
    from gpuschedule_b200 import flags
    F = flags.define_simulator_flags()
    F.reset(["--num_switch", "4", "--enable_network_costs", "False", "--schedule", "fifo", "--nopack"])
    assert F.num_switch == 4 and F.enable_network_costs is False and F.pack is False
    assert F.num_gpu_p_node == 8 and F.mem_p_node == 512 and F.bandwidth == 1250
    F.reset(["--enable_network_costs"])
    assert F.enable_network_costs is True


def test_log_manager_headers_and_object_api(tmp_path):
    from gpuschedule_b200 import log_manager

    class Infra:
        nodes = {str(i): None for i in range(3)}

        def get_total_gpus(self):
            return 6

    class F:
        scheme = "yarn"

    lm = log_manager.LogManager(str(tmp_path), F())
    lm.init(Infra())
    assert open(tmp_path / "cpu.csv", newline="").read() == "time,cpu0,cpu1,cpu2\r\n"
    assert open(tmp_path / "gpu.csv", newline="").read() == "time,gpu0,gpu1,gpu2,gpu3,gpu4,gpu5\r\n"
    assert open(tmp_path / "network.csv", newline="").read() == "time,in0,out0,in1,out1,in2,out2\r\n"
    assert open(tmp_path / "memory.csv", newline="").read() == "time,max,99th,95th,med\r\n"
    lm.step_cluster(log_manager.LogInfo(3, 0, 0, 6, 0.0, 0.0, 0.0, float("nan"), 0, 0, 0, 0), 1)
    lines = open(tmp_path / "cluster.csv", newline="").read().split("\r\n")
    assert lines[1] == "1,3,0,0,6,0.0,0.0,0.0,nan,0,0,0,0"


def test_bracketed_float_text_is_numpy_array_text():
    """rngcol._format_bracketed prints with C's %.8f; the reference prints str(np.array([v])) (dragon4, precision 8,
    unique): same text on random values of every magnitude the column takes, short decimals and binary ties."""
    from gpuschedule_b200 import rngcol
    rng = np.random.default_rng(5)
    vals = [0.0, 2.0 ** -9, 3 * 2.0 ** -9, 5 * 2.0 ** -9, 2.0 ** -13, 0.5, 1.0, 100.0, 12345678.0, 1e-5, 3e-7, 1e8, 2.5e9, 99.99999999, 0.000100001]
    for scale in (1e-3, 0.05, 1.0, 7.0, 100.0, 1e4, 1e7):
        vals += (rng.random(20000) * scale).tolist() + np.round(rng.random(5000) * scale, 8).tolist() + np.round(rng.random(5000) * scale, 3).tolist()
        vals += ((rng.integers(1, 1 << 20, 5000) / 1024.0) * scale).tolist()
    text = rngcol._format_bracketed(np.array(vals))
    for v, t in zip(vals, text):
        assert t == str(np.array([v])), (v, t)


def test_logcol_walk_matches_a_direct_numpy_walk():
    """gs_logcol_* (host helper of the log writer) against the definition: per row, busy devices in key order, one value each"""
    from gpuschedule_b200 import capi
    rng = np.random.default_rng(11)
    n_rows, width, njobs = 300, 96, 40
    loc, scale = rng.random(njobs) * 90 + 5, rng.random(njobs) * 20
    # holdings that never overlap on a device: consecutive intervals per device
    first, last, key, job = [], [], [], []
    for k in range(width):
        r = int(rng.integers(0, 50))
        while r < n_rows + 20:
            ln = int(rng.integers(1, 60))
            if rng.random() < 0.7:
                first.append(r); last.append(r + ln - 1); key.append(k); job.append(int(rng.integers(0, njobs)))
            r += ln + int(rng.integers(0, 3))
    order = np.argsort(np.array(first), kind="stable")
    first, last = np.array(first, dtype=np.int64)[order], np.array(last, dtype=np.int64)[order]
    key, job = np.array(key, dtype=np.int32)[order], np.array(job, dtype=np.int32)[order]
    owner = np.full((n_rows, width), -1)
    for f, l, k, j in zip(first, last, key, job):
        owner[f:min(l, n_rows - 1) + 1, k] = j
    with capi.LogColumn(n_rows, width, first, last, key, job) as col:
        counts = col.counts()
        assert np.array_equal(counts, (owner >= 0).sum(axis=1))
        z = rng.standard_normal(int(counts.sum()))
        half = n_rows // 3
        a1, u1 = col.rows(half, loc, scale, z[:int(counts[:half].sum())])
        a2, u2 = col.rows(n_rows, loc, scale, z[int(counts[:half].sum()):])
    acc, unc = np.concatenate([a1, a2]), np.concatenate([u1, u2])
    p = 0
    for r in range(n_rows):
        a, nu = 0.0, 0
        for k in range(width):
            j = owner[r, k]
            if j < 0:
                continue
            x = float(loc[j]) + float(scale[j]) * float(z[p]); p += 1
            if x >= 100.0:
                a += 100.0
            else:
                a += x; nu += 1
        assert a == acc[r] and nu == unc[r], r
    with pytest.raises(capi.GsError):                       # unsorted holdings are refused
        capi.LogColumn(n_rows, width, first[::-1].copy(), last[::-1].copy(), key, job)


def test_parsed_trace_cache_round_trip_and_invalidation(tmp_path):
    import time as _time
    from gpuschedule_b200 import ingest, tracegen
    p = str(tmp_path / "t.csv")
    cache = str(tmp_path / "cache")
    tracegen.write_trace(p, 3000, seed=3, rate=0.5)
    a = ingest.load_table(p, 0.5, cache)
    assert len(os.listdir(cache)) == 1
    b = ingest.load_table(p, 0.5, cache)                    # served from the cache
    plain = ingest.JobTraceReader(p).prepare_jobs().table(0.5)
    for t in (a, b):
        for k in ingest._ARRAY_FIELDS:
            assert getattr(t, k).dtype == getattr(plain, k).dtype and getattr(t, k).tobytes() == getattr(plain, k).tobytes(), k
        assert t.label == plain.label and t.num_gpu_text == plain.num_gpu_text and t.n == plain.n
        assert t.extra["mem_avg_mib"].tobytes() == plain.extra["mem_avg_mib"].tobytes()
    ingest.load_table(p, 1.0, cache)                        # another scale factor: another entry
    assert len(os.listdir(cache)) == 2
    _time.sleep(0.01)
    tracegen.write_trace(p, 3001, seed=4, rate=0.5)         # the file changed: a miss, and the new contents
    c = ingest.load_table(p, 0.5, cache)
    assert c.n == ingest.JobTraceReader(p).prepare_jobs().table(0.5).n and len(os.listdir(cache)) == 3
    assert ingest.load_table(p, 0.5, None).n == c.n         # no cache directory: plain parse
