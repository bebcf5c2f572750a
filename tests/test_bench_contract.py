"""bench.py's reference arm runs without a GPU: check the JSON line it prints against the driver's contract
(keys, types, the tier's extra objects).  Small workload so it stays in the CPU suite's budget."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytest.importorskip("cv2")


def test_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                        "--warmup", "0", "--units", "2", "--features", "300", "--width", "640", "--height", "240", "--cpu-seconds", "2"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "frames" in cb["sample"]
    assert "workload" in d["config"] and "model" not in d["config"]
    # both ways of running the CPU path are always reported, each as median / min / max of 3 repetitions
    seq, pool = cb["sequential"], cb["pool"]
    assert seq["reps"] == 3 and seq["min"] <= seq["median"] <= seq["max"] and seq["seconds"] >= 1.9
    assert "error" in pool or (pool["reps"] == 3 and pool["min"] <= pool["median"] <= pool["max"] and pool["busy_workers"] >= 1)
    assert cb["value"] == max(seq["median"], pool.get("median", 0.0))


def test_non_rank0_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_native_gather_bookkeeping_never_exceeds_the_library_depth():
    """bench.NativeGather (host side of the C-ABI record gather): posts every step, harvests the oldest table only when
    VO_DIST_DEPTH posts are outstanding, drains in order -- checked against a stub context that enforces the library's rule."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from visual_odom_b200.capi import VO_DIST_DEPTH

    class Stub:
        def __init__(self):
            self.posted, self.waited, self.max_out = 0, 0, 0

        def dist_gather_post(self, slot, n):
            assert self.posted - self.waited < VO_DIST_DEPTH, "the library would refuse this post"
            self.posted += 1
            self.max_out = max(self.max_out, self.posted - self.waited)

        def dist_gather_wait(self, n, raw=False):
            assert self.waited < self.posted and raw
            self.waited += 1
            return self.waited - 1

    ctx = Stub()
    g = bench.NativeGather(ctx, 8)
    assert g.DEPTH == VO_DIST_DEPTH
    for s in range(20):
        g.post_step((s % 3) * 8, None, None)
    tables = g.drain()
    assert tables == list(range(20)) and ctx.posted == ctx.waited == 20 and ctx.max_out == VO_DIST_DEPTH
    assert g.drain() == []


def test_dump_outputs_writes_float_arrays_within_the_budget(tmp_path):
    """bench.dump_outputs (--dump-outputs DIR): float32 / float64 .npy files only, the point lists concatenated in unit order
    as the records count them, and a step whose worst case exceeds the budget cut to the same seeded sample of units."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    rng = np.random.default_rng(5)
    recs, outs = [], []
    for u in range(40):
        nv = int(rng.integers(0, 50))
        ni = int(rng.integers(0, nv + 1))
        recs.append(dict(n_features=50, n_detected=60 + u, n_tracked=nv + 1, n_valid=nv, n_inliers=ni, ransac_iters=u, pnp_status=0,
                         rvec=rng.normal(size=3), tvec=rng.normal(size=3), R=rng.normal(size=(3, 3))))
        outs.append(dict(l0=rng.random((nv, 2), np.float32), r0=rng.random((nv, 2), np.float32), l1=rng.random((nv, 2), np.float32),
                         r1=rng.random((nv, 2), np.float32), X=rng.random((nv, 3), np.float32),
                         kept_idx=np.sort(rng.choice(50, nv, replace=False)).astype(np.int32), inliers=np.arange(ni, dtype=np.int32)))

    def load(d):
        files = sorted(os.listdir(d))
        assert all(f.endswith(".npy") for f in files)
        return {f[:-4]: np.load(os.path.join(d, f)) for f in files}

    bench.dump_outputs(str(tmp_path / "all"), recs, recs, outs, 50)
    a = load(tmp_path / "all")
    names = {"units"} | {p + k for p in ("resident_", "e2e_") for k in ("counts", "rvec", "tvec", "R")} | {"e2e_" + k for k, _ in bench.POINT_LISTS}
    assert set(a) == names and all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert np.array_equal(a["units"], np.arange(40)) and a["e2e_counts"].shape == (40, 7) and a["e2e_R"].shape == (40, 3, 3)
    assert np.array_equal(a["resident_counts"][:, 3], [r["n_valid"] for r in recs])
    for k, dt in bench.POINT_LISTS:
        assert np.array_equal(a["e2e_" + k], np.concatenate([o[k] for o in outs]).astype(dt)), k

    bench.DUMP_BYTES = 10 * (60 * 50 + 360)         # room for the worst case of 10 units
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), recs, recs, outs, 50)
    s1, s2 = load(tmp_path / "s1"), load(tmp_path / "s2")
    assert all(np.array_equal(s1[k], s2[k]) for k in names)
    units = s1["units"].astype(int)
    assert len(units) == 10 and np.all(np.diff(units) > 0) and sum(x.nbytes for x in s1.values()) <= bench.DUMP_BYTES
    assert np.array_equal(s1["e2e_tvec"], [recs[u]["tvec"] for u in units])
    assert np.array_equal(s1["e2e_l1"], np.concatenate([outs[u]["l1"] for u in units]))
