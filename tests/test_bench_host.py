"""CPU: host-side pieces of the measurement contract that need no device -- the reference arm's rank rule under torchrun,
the launch-list summariser, and the growth-scaled CPU baseline of the bench line."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_other_ranks_exit_silently():
    """`bench.py --impl reference` under torchrun: rank 0 alone measures and prints; the others exit 0 without work"""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2",
                        "--warmup", "1"], env=env, capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_launch_list_summary(tmp_path):
    src = os.path.join(ROOT, "profiles", "r2_launches_one_draw_final.csv")
    out = tmp_path / "s.json"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "launch_list_summary.py"), src, str(out), "cmd", "note"],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    s = json.load(open(out))
    k = s["kernels"]
    assert s["launches_in_window"] == sum(v["launches"] for v in k.values()) == 620
    assert abs(sum(v["share"] for v in k.values()) - 1.0) < 1e-12
    top = next(iter(k))
    assert "oz_mma_kernel" in top and k[top]["share"] > 0.35          # the int8 tcgen05 GEMM leads the serialised list too
    assert any("potrf_diag_kernel" in n for n in k) and any("oz_slice_kernel" in n for n in k)


def test_cpu_baseline_scales_by_measured_growth(monkeypatch):
    """the bench line's CPU baseline: largest N within the budget, scaled to N = 16384 by the growth per doubling it
    measured itself (not by the cubic flop count)"""
    sys.path.insert(0, ROOT)
    import bench
    import oracle
    cost = {1024: 0.01, 2048: 0.05, 4096: 0.2, 8192: 0.8, 16384: 3.0}       # seconds a fake host needs: growth 4x, then 3.75x
    clock = {"t": 0.0}

    def fake(X, y, Xn, params, kind, jitter=1e-6):
        clock["t"] += cost[X.shape[0]]
    monkeypatch.setattr(oracle, "exact_posterior", fake)
    monkeypatch.setattr(oracle, "exact_posterior_chol", fake)
    monkeypatch.setattr(bench.time, "perf_counter", lambda: clock["t"])
    small = {k: v for k, v in bench.WORKLOAD.items()}
    out = bench.cpu_baseline(budget_s=1.0)
    # budget 1 s: 4096 -> predicted 0.8 fits -> runs 8192 (0.8 s); next predicted 3.2 s does not -> scaled by 0.8/0.2 = 4
    assert "N=8192" in out["sample"] and "4.00x" in out["sample"]
    assert abs(1.0 / out["value"] - 3.2) < 1e-9
    # the Cholesky formulation gets half the budget: stays at 4096 (predicted 0.8 > 0.5), two doublings at 4x
    assert "N=4096" in out["best_cpu_formulation"]["sample"]
    assert abs(1.0 / out["best_cpu_formulation"]["value"] - 0.2 * 16) < 1e-9
    assert bench.WORKLOAD == small


def test_dump_outputs_writes_all_or_a_seeded_sample(tmp_path, monkeypatch):
    """--dump-outputs: every draw while the arrays fit the limit; above it the same seeded rows of each array, bounded"""
    sys.path.insert(0, ROOT)
    import bench
    S, P = 40, 16
    mean = np.arange(S * P, dtype=np.float64).reshape(S, P)
    var = mean + 0.5
    bench.dump_outputs(str(tmp_path / "all"), {"mean": mean, "var": var})
    assert sorted(os.listdir(tmp_path / "all")) == ["mean.npy", "var.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "mean.npy"), mean)
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "var.npy"), var)

    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * (2 * P * 8 + 8))        # room for 10 of the 40 draws
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"mean": mean, "var": var}, "_rank1")
    assert sorted(os.listdir(tmp_path / "a")) == ["draws_rank1.npy", "mean_rank1.npy", "var_rank1.npy"]
    rows = np.load(tmp_path / "a" / "draws_rank1.npy")
    assert rows.dtype == np.float64 and rows.shape == (10,) and len(set(rows)) == 10
    r = rows.astype(int)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "mean_rank1.npy"), mean[r])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "var_rank1.npy"), var[r])
    np.testing.assert_array_equal(np.load(tmp_path / "b" / "draws_rank1.npy"), rows)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_LIMIT_BYTES + 3 * 128
