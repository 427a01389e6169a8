"""bench.py contract pieces that can be checked without a GPU: the reference arm prints ONE JSON line with the agreed keys,
and the product arm fails loudly (no JSON, non-zero exit) when there is no device -- there is no CPU fallback."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _run(args, timeout=600):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    p = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GFLOPS" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "4096" in d["metric"] and "sample" in d["cpu_baseline"]


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = _run(["--steps", "1", "--warmup", "0", "--no-cpu"], timeout=300)
    assert p.returncode != 0
    assert not [l for l in p.stdout.splitlines() if l.strip().startswith("{")]


@pytest.mark.parametrize("args,msg", [(["--steps", "0"], "--steps must be at least 1"),
                                      (["--impl", "reference", "--dump-outputs", "x"], "--impl reference has none")])
def test_invalid_arguments_are_refused(args, msg):
    p = _run([*args, "--warmup", "0", "--no-cpu"], timeout=300)
    assert p.returncode == 2 and msg in p.stderr


def test_dump_sample_within_budget_over_ranks():
    """--dump-outputs' row sample (the seeded branch the default 4096^2 run takes), its budget split over the ranks: rows and
    index of all ranks together within the budget, rows sorted and unique, the same on every call, and they are C's rows."""
    import numpy as np
    import torch
    import bench
    M, N, budget = 1000, 300, 256 << 10
    for world in (1, 3, 4):
        total = 0
        for rank in range(world):
            C = torch.randn(M * N, generator=torch.Generator().manual_seed(rank))
            idx, rows = bench.sample_rows(C, M, N, budget // world)
            idx2, rows2 = bench.sample_rows(C, M, N, budget // world)
            assert np.array_equal(idx, idx2) and np.array_equal(rows, rows2)
            assert idx.dtype == np.float64 and rows.dtype == np.float32 and 0 < len(idx) < M
            assert np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < M and np.array_equal(idx, np.round(idx))
            assert np.array_equal(rows, C.numpy().reshape(N, M).T[idx.astype(np.int64)])
            total += idx.nbytes + rows.nbytes
        assert total <= budget, world
    with pytest.raises(ValueError):
        bench.sample_rows(C, M, N, 4 * N)  # not even one row and its index entry
    n = 4096  # the default size on 1, 2 and 8 ranks stays within the budget in all
    C = torch.zeros(n * n)
    for world in (1, 2, 8):
        idx, rows = bench.sample_rows(C, n, n, bench.DUMP_BYTES // world)
        assert world * (idx.nbytes + rows.nbytes) <= bench.DUMP_BYTES < 64e6 and len(idx) < n


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(cuda, oracle, tmp_path):
    """--dump-outputs DIR: two runs with the same arguments dump the same C, and it is the C the timed path leaves --
    (warmup + steps) applications of C = A*B^T - 1.5*C from C = 0 -- against the TF32 model on the bench's own inputs;
    --steps K times exactly K steps."""
    import numpy as np
    import bench
    n, steps = 1024, 3
    dumps = []
    for i in range(2):
        p = _run(["--size", str(n), "--steps", str(steps), "--warmup", "1", "--no-sweep", "--no-cpu", "--strong-size", "0",
                  "--dump-outputs", str(tmp_path / str(i))])
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads([l for l in p.stdout.splitlines() if l.strip()][-1])
        assert d["steps"] == steps and d["gpu_launches"] in (steps, 2 * steps)  # (small sizes: the encode is a launch of its own)
        idx, rows = np.load(tmp_path / str(i) / "C_row_index.npy"), np.load(tmp_path / str(i) / "C_rows.npy")
        assert idx.dtype == np.float64 and rows.dtype == np.float32 and rows.shape == (n, n)
        assert np.array_equal(idx, np.arange(n))  # 4 MiB: every row
        dumps.append(rows)
    assert np.array_equal(dumps[0], dumps[1])
    g = cuda.Generator(device="cuda").manual_seed(1234)  # bench.py's inputs on rank 0
    A = bench.fill_ref_dist(cuda.empty(n * n, device="cuda"), g).cpu().numpy()
    B = bench.fill_ref_dist(cuda.empty(n * n, device="cuda"), g).cpu().numpy()
    P = oracle.as2d(oracle.sgemm_nt_tf32_model(n, n, n, 1.0, A, B, 0.0, np.zeros(n * n, np.float32)), n, n)
    want = P.astype(np.float64) * sum((-1.5) ** j for j in range(d["warmup"] + steps))
    assert np.linalg.norm(dumps[0] - want) / np.linalg.norm(want) < 1e-4


def test_committed_product_line_has_the_contract_keys():
    """The product arm cannot run here (no GPU); the line it printed on the round's last box is committed under profiles/ --
    check that artefact against the contract, so that a key dropped from bench.py's output is noticed on the CPU side too."""
    d = json.loads((ROOT / "profiles" / "r02_bench_n1_final.json").read_text().strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "clocks", "gpu_launches", "sweep", "parity", "abft"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 20 and d["gpu_launches"] == d["steps"] and d["higher_is_better"] is True
    assert "workload" in d["config"] and "model" not in d["config"]
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3 and r["traffic"] > 0
    assert 0.5 < r["frac"] < 1.0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 3 * 4 * 4096 * 4096 and e["d2h_bytes_per_step"] == 4 * 4096 * 4096 and 0 < e["value"] < d["value"]
    assert d["clocks"]["sm_mhz"] > 0 and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert d["parity"]["ok"] and d["parity"]["rel_fro"] < d["parity"]["tolerance"] == 1e-3
    sizes = [row["n"] for row in d["sweep"]]
    assert sizes == list(range(1024, 16385, 1024))
    for row in d["sweep"]:
        assert {"abft_gflops", "plain_gflops", "cublas_tf32_gflops", "overhead_pct_vs_cublas_tf32"} <= set(row)
    # the claim DESIGN.md / README.md make about this line
    assert d["abft"]["overhead_pct_vs_cublas_tf32"] <= 10.0
    assert all(row["overhead_pct_vs_cublas_tf32"] <= 11.0 for row in d["sweep"] if row["n"] >= 4096)
