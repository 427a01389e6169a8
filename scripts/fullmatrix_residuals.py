#!/usr/bin/env python
"""Whole-matrix residuals of the fused ABFT kernel against the float64 reference (oracle/fullref.py), one JSON line per
case on stdout: max |got - ref| / (|alpha| * S) over every element, the kernel's own fault-free row residual
stats.max_rel_residual (|d1| / sum|acc|, the quantity the detection threshold tau_rel = 1e-5 is compared with), the eps the
tests use for that case, and what was flagged.  The first line names the card, its power limit and SM clock limit.

  python scripts/fullmatrix_residuals.py [--quick] > profiles/r03_fullmatrix_residuals.jsonl

Cases: bench.py's sweep (1024 .. 16384, ids 40 / resolved, reference distribution, alpha = 1, beta = -1.5), the ragged /
multi-wave shapes of tests/test_gpu_fullmatrix.py, and four input distributions (reference, N(0,1), U[0,1), 2^+-20 row
scales) at 2048^3, 4096^3 (ids 31, 16) and (1024, 1024, K) for K = 16384, 32768, 65536 (id 31).
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import __graft_entry__ as ge  # noqa: E402
from oracle import fullref as R  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="skip 16384^3 and K = 65536")
    args = ap.parse_args()
    ft = ge.load_package()
    torch.cuda.set_device(0)
    h = ft.FtSgemm()
    print(json.dumps({"card": card(), "torch": torch.__version__, "note": "name, power.limit, clocks.max.sm"}), flush=True)

    def case(tag, M, N, K, kid, dist, alpha=1.0, beta=-1.5):
        g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
        A = R.fill(torch.empty(M * K, device="cuda"), dist, g, M, K)
        B = R.fill(torch.empty(N * K, device="cuda"), dist, g, N, K)
        C0 = torch.randn(M * N, generator=g, device="cuda")
        ref = R.Reference(M, N, K, A, B, C0, alpha, beta)
        C = C0.clone()
        h.stats()
        h.run(kid, M, N, K, A, B, C, alpha, beta, None)
        st = h.stats()
        eps = R.eps_for(K, dist)
        nbad = int(ref.bad_mask(C, eps).sum())
        line = {"case": tag, "M": M, "N": N, "K": K, "id": kid, "resolved_id": ft.select_kernel(M, N, K, True) if kid == 40 else kid,
                "dist": dist, "max_ratio_to_S": ref.max_ratio(C), "max_rel_residual": st["max_rel_residual"],
                "max_abs_residual": st["max_abs_residual"], "detected": st["detected"], "eps": eps, "failing_elements": nbad}
        print(json.dumps(line), flush=True)
        del A, B, C0, C, ref
        torch.cuda.empty_cache()

    for i in range(1, 17):
        n = 1024 * i
        if args.quick and n == 16384:
            continue
        case("sweep", n, n, n, ft.ID_ABFT_AUTO, "ref")
    for (M, N, K), kid in (((4100, 4196, 4127), 31), ((4096, 4064, 4096), 31), ((4096, 4100, 4096), 31),
                           ((3072, 3072, 3072), 31), ((2052, 12288, 1000), 31), ((12288, 2052, 1000), 31),
                           ((6144, 6144, 12288), 31), ((12292, 12292, 1100), 31), ((256, 65536, 1024), 31),
                           ((65536, 256, 1024), 31), ((1024, 1024, 65536), 32)):
        if args.quick and K == 65536:
            continue
        case("ragged", M, N, K, kid, "ref")
    for dist in ("ref", "normal", "uniform01", "wide"):
        for (M, N, K), kid in (((2048, 2048, 2048), 31), ((2048, 2048, 2048), 16), ((4096, 4096, 4096), 31),
                               ((4096, 4096, 4096), 16), ((1024, 1024, 16384), 31), ((1024, 1024, 32768), 31),
                               ((1024, 1024, 65536), 31)):
            if args.quick and K == 65536:
                continue
            case("distribution", M, N, K, kid, dist)
    h.close()


if __name__ == "__main__":
    main()
