"""bench.py pieces that run without a GPU: the `roofline` object arithmetic and
the reference arm (the CPU port timed on the host cores), which must print
one JSON line; on a GPU, the step count and `--dump-outputs`."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_roofline_object_single_kernel_step():
    bench = _bench()
    # 1000 bracketed launches of ~72 us; region 1: 1000 steps in 67.5 ms, one launch per step
    times = np.full(1000, 0.072, dtype=np.float32)
    times[:10] = 0.0698
    prof = {0: (float(times.astype(np.float64).sum()), 1000), 1: (0.0, 0), 2: (0.0, 0), 3: (0.0, 0)}
    pt = {0: times, 1: np.zeros(0, np.float32), 2: np.zeros(0, np.float32)}
    r = bench.roofline_object(prof, pt, 67.5, 1000, 1000, "product", 10_000_000, 320e6, 6576.1,
                              "measured", "config5_10M_product_50k_tokens", False)
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["kernel"].startswith("product_sweep_tma")
    # traffic: only from an ncu capture of THIS kernel on THIS workload (profiles/traffic.json), else null
    assert r["traffic"] == bench.read_traffic("config5_10M_product_50k_tokens", "product_sweep_tma")
    assert bench.read_traffic("config2_100k_product_1k_tokens", "sweep_kernel_univ3") is None
    assert r["l2_state"] == "inputs larger than L2"
    assert abs(r["avg_launch_us"] - 71.978) < 0.01
    assert abs(r["achieved"] - 320e6 / (r["avg_launch_us"] * 1e-6) / 1e9) < 1e-6
    assert abs(r["frac"] - r["achieved"] / 6576.1) < 1e-12
    assert r["launch_us"]["min"] < r["launch_us"]["median"] <= r["launch_us"]["p95"] <= r["launch_us"]["max"]
    b = r["back_to_back"]
    assert abs(b["launch_us"] - 67.5) < 1e-9 and abs(b["achieved"] - 4740.74) < 0.01
    assert b["frac"] > r["frac"]            # overlap of consecutive launches; never the headline
    assert "exchange_avg_us" not in r
    json.dumps(r)                           # plain Python types only


def test_roofline_object_mixed_and_exchange():
    bench = _bench()
    prof = {0: (10.0, 100), 1: (30.0, 100), 2: (0.0, 0), 3: (1.2, 100)}
    pt = {0: np.full(100, 0.1, np.float32), 1: np.full(100, 0.3, np.float32), 2: np.zeros(0, np.float32)}
    r = bench.roofline_object(prof, pt, 45.0, 100, 300, "mixed", 1_000_000, 40e6, 6650.0, "fallback",
                              "config3_1M_mixed_10k_tokens", True)
    assert r["l2_state"].startswith("flushed")
    assert r["kernel"].startswith("product_sweep_tma<GeometricMeanTwoCoin>")
    assert r["algorithmic_bytes_per_launch"] == 500_000 * 48
    assert "back_to_back" not in r          # several launches per step: no single-kernel figure
    assert abs(r["exchange_avg_us"] - 12.0) < 1e-9
    assert r["traffic"] == bench.read_traffic("config3_1M_mixed_10k_tokens", "product_sweep_tma_geomean")
    r2 = bench.roofline_object(prof, pt, 45.0, 100, 300, "mixed", 1_000_000, 40e6, 6650.0, "fallback",
                               "some_other_workload", True)
    assert r2["traffic"] is None            # no capture of that workload: no number


def test_reference_arm_prints_contract_line():
    """`bench.py --impl reference` (the CPU port on the host cores) on a tiny budget."""
    env = dict(os.environ, OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "2", "--warmup", "1", "--workload", "config2_100k_product_1k_tokens"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    r = json.loads(lines[0])
    assert r["impl"] == "reference" and r["n_gpus"] == 1 and r["higher_is_better"] is True
    assert r["metric"] and r["unit"] == "pools/s" and r["value"] > 0 and r["steps"] == 2
    assert r["cpu_baseline"]["kind"] == "port" and r["cpu_baseline"]["cores"] >= 1
    assert r["e2e"]["value"] == r["value"] and r["e2e"]["h2d_bytes_per_step"] == 0


@pytest.mark.gpu
def test_dump_outputs_is_the_timed_sweep(oracle, synth, tmp_path):
    """`--steps K` times K sweeps (one launch each), and `--dump-outputs` writes the [Ψ; acc]
    the last of them computed: the CPU oracle's fold of the same seeded pools at the same ν."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "7", "--warmup", "2",
                          "--workload", "config2_100k_product_1k_tokens", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path / "out")],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert r["steps"] == 7 and r["gpu_launches"] == 7 and r["e2e"]["steps"] == 7 and "sustained" not in r
    psi, acc = np.load(tmp_path / "out" / "psi.npy"), np.load(tmp_path / "out" / "acc.npy")
    n = 1_000
    assert psi.dtype == np.float64 and psi.shape == (n,) and acc.shape == (1,)
    R, g, Ai = synth.product_pools(100_000, n, seed=1234)
    v = synth.dual_prices(n, "near")
    D, L = oracle.sweep_product(R, g, Ai, v, threads=8)
    accx, Gx, absG = oracle.fold_compensated(Ai, D, L, v, n)
    slack, S, deg = np.zeros(n), np.zeros(n), np.zeros(n)  # economized math + fixed-point slice quantum,
    for side in (0, 1):                                    # as bench.verify_reduction bounds them
        np.add.at(slack, Ai[:, side] - 1, 32 * np.finfo(float).eps * (R[:, 0] + R[:, 1]) / g)
        np.add.at(S, Ai[:, side] - 1, R[:, side])
        np.add.at(deg, Ai[:, side] - 1, 1.0)
    slack += deg * S * 2.0 ** -53
    assert np.all(np.abs(psi - Gx.astype(np.float64)) <= 1e-12 * absG + slack)
    assert abs(acc[0] - float(accx)) <= 1e-12 * float(np.sum(absG * v)) + float(np.sum(slack * v))
