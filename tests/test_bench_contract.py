"""bench.py contract (CPU part): the reference arm prints ONE JSON line with the required keys, and the
algorithmic-flop helper matches N^3/3 to leading order."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout + r.stderr
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is False and d["unit"] == "ms" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"] and "C4" in d["config"]["workload"]  # the same workload as the GPU arm at every N
    assert "extrapolated" in d["cpu_baseline"]["sample"]  # bounded N = 8192 sample, labelled


def test_trailing_flops_close_to_third_n_cubed():
    sys.path.insert(0, ROOT)
    import bench
    for n in (4096, 32768):
        assert abs(bench.trailing_flops(n) / (n ** 3 / 3.0) - 1.0) < 0.06
    assert abs(bench.trailing_flops(65536, 512) / (65536 ** 3 / 3.0) - 1.0) < 0.03


def test_reference_arm_other_workloads_are_bounded():
    """C2 runs in full; C3 / C5 samples are bounded and labelled"""
    sys.path.insert(0, ROOT)
    import bench
    cfg, scale, sample = bench.cpu_sample("C2", 4096)
    assert scale == 1.0 and cfg["X"].shape == (4096, 8)
    cfg, scale, sample = bench.cpu_sample("C5", 1000000)
    assert cfg["X"].shape[0] == 20000 and scale > 100 and "extrapolated" in sample
    cfg, scale, sample = bench.cpu_sample("C3", 16384)
    assert cfg["X"].shape[0] == 8192 and abs(scale - 8.0) < 1e-9 and cfg["Xs"].shape[0] == 5000


def test_roofline_traffic_record_is_committed():
    """bench.py fills roofline.traffic from the committed ncu capture of the benched workload (profiles/traffic.json)"""
    sys.path.insert(0, ROOT)
    import bench
    for wl in ("C4", "C4h"):
        t = bench.ncu_traffic(wl)
        assert t and t["dram_bytes_per_launch"] > 0 and t["algorithmic_bytes_per_launch"] > 0
        assert 1.0 <= t["ratio"] < 1.5, t["ratio"]          # traffic close to the algorithmic bytes: no wasted re-reads
        assert os.path.exists(os.path.join(ROOT, t["capture"]))


def test_dump_outputs_fits_budget_with_a_fixed_sample(tmp_path):
    """--dump-outputs: one float .npy per output, all of them within DUMP_BYTES; an oversized output is replaced by the
    same seeded sample of its entries on every run"""
    sys.path.insert(0, ROOT)
    import bench
    outs = {"logpdf": np.array([-1.5]), "alpha": np.arange(bench.DUMP_BYTES // 8 + 10, dtype=np.float64)}
    for d in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / d))
    sizes = [os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")]
    assert sorted(os.listdir(tmp_path / "a")) == ["alpha.npy", "logpdf.npy"] and sum(sizes) <= bench.DUMP_BYTES
    a, b = np.load(tmp_path / "a" / "alpha.npy"), np.load(tmp_path / "b" / "alpha.npy")
    assert a.dtype == np.float64 and 0 < a.size < outs["alpha"].size and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0)  # sampled entries keep their order
    assert np.load(tmp_path / "a" / "logpdf.npy").tolist() == [-1.5]


@pytest.mark.gpu
def test_dump_outputs_match_oracle(tmp_path, ref):
    """bench.py --dump-outputs on C2 writes the logpdf and alpha of its last timed step; they match the oracle"""
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C2", "--steps", "2", "--warmup", "1",
                        "--quick", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    cfg = ref.make_config("C2")
    lp = np.load(out / "logpdf.npy")
    alpha = np.load(out / "alpha.npy")
    lp_ref = ref.logpdf(cfg["k"], cfg["mean"], cfg["noise"], cfg["X"], cfg["y"])
    alpha_ref = ref.posterior(cfg["k"], cfg["mean"], cfg["noise"], cfg["X"], cfg["y"])["alpha"]
    assert lp.dtype == np.float64 and lp.shape == (1,) and abs(lp[0] - lp_ref) <= 1e-8 * abs(lp_ref)
    assert alpha.shape == (4096,) and np.allclose(alpha, alpha_ref, rtol=1e-7, atol=1e-9)
