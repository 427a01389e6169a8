"""Generate tests/golden/*.json from the reference's OWN code: oracle/_ref/libref_utils.so (its utils/utils.cu compiled
unmodified) and oracle/_ref/libref_kernels_cpu.so (its generated kernels under the CPU thread shim).  Run where the
reference sources are available to `make -C oracle`; the tests read only the JSON.

ref_cpu_gemm.json, for END in {64,128,160,256,512,1024}: srand(10); A,B,C = generate_random_matrix(END); C=0
(sgemm.cu:12,52-56); C = cpu_gemm(1, 0, B^T-buffer, A-buffer) which is the kernels' column-major NT result
(SURVEY.md section 8c oracle 1).  Stored: leading elements of A/B/C, selected C entries, sums, and a
sha256 of the raw float32 bytes of A, B and C.

ref_checks.json: the verdicts of the reference's verify_matrix on the END = 160 product, and the output of each
generated kernel that tests/test_oracle.py::test_reference_kernels_on_cpu names, on that test's inputs: a sha256 of its
float32 bytes plus the elements where it differs from the sequential-k oracle product (the injected-and-corrected ones).
"""
import hashlib, json, sys
from pathlib import Path
import numpy as np
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from oracle import oracle as O


def sha(a):
    return hashlib.sha256(a.tobytes()).hexdigest()


out_dir = Path(__file__).resolve().parents[1] / "tests" / "golden"
out_dir.mkdir(parents=True, exist_ok=True)
r = O.ref_utils()
assert r is not None, "needs oracle/_ref (run `make -C oracle`)"
gold = {}
for n in (64, 128, 160, 256, 512, 1024):
    A, B, C = O.ref_make_inputs(n)
    # cpu_gemm is row-major square: Z = X*Y.  With X := B-buffer read row-major = B^T ... see SURVEY 8c:
    # kernels' C buffer == cpu_gemm(alpha, beta, B^T_buffer, A_buffer).  B^T_buffer: row-major (K x N)^T
    # Concretely Cbuf[m + n*M] = sum_k A[m+k*M]*B[n+k*N]; as row-major Z[i=n][j=m] = sum_k X[n][k] Y[k][m]
    # with X[n][k] = B[n + k*N] (i.e. X = transpose of the B buffer read row-major) and Y = A buffer row-major.
    X = np.ascontiguousarray(B.reshape(n, n).T)
    Z = np.zeros(n * n, np.float32)
    r.ref_cpu_gemm(1.0, 0.0, O._p(X.reshape(-1)), O._p(A), n, O._p(Z))
    gold[str(n)] = {
        "A_head": [float(x) for x in A[:8]], "B_head": [float(x) for x in B[:8]],
        "C_sel": {"0": float(Z[0]), "1": float(Z[1]), str(n): float(Z[n]), str(n * n - 1): float(Z[n * n - 1])},
        "C_sum": float(Z.astype(np.float64).sum()), "C_abs_sum": float(np.abs(Z.astype(np.float64)).sum()),
        "sha256": {"A": sha(A), "B": sha(B), "C": sha(Z)},
    }
    print(n, gold[str(n)]["C_sel"], gold[str(n)]["C_sum"], gold[str(n)]["C_abs_sum"])
    if n == 160:
        bad = Z.copy()
        bad[77] += 5.0
        verify_160 = {"identical": int(r.ref_verify_matrix(O._p(Z), O._p(Z.copy()), n, n)),
                      "element_77_plus_5": int(r.ref_verify_matrix(O._p(Z), O._p(bad), n, n))}
(out_dir / "ref_cpu_gemm.json").write_text(json.dumps(gold, indent=1) + "\n")

rk = O.ref_kernels()
assert rk is not None, "needs oracle/_ref/libref_kernels_cpu.so (run `make -C oracle`)"
kernels = {}
for kid, variant, K in ((6, "huge", 160), (16, "huge", 160), (13, "large", 160), (11, "small", 480)):
    M, N = O.VARIANTS[variant][:2]
    rng = np.random.default_rng(2)
    A = (rng.integers(-9, 10, M * K) * 0.1).astype(np.float32)
    B = (rng.integers(-9, 10, N * K) * 0.1).astype(np.float32)
    pad = np.zeros(4096, np.float32)  # the kernels' last loads run past the end of A and B
    Ap, Bp = np.concatenate([A, pad]), np.concatenate([B, pad])
    C = np.zeros(M * N, np.float32)
    assert rk.ref_kernel_run(kid, M, N, K, O._p(Ap), O._p(Bp), O._p(C), 1.0, 0.0) == 0
    plain = O.sgemm_nt(M, N, K, 1.0, A, B, 0.0, np.zeros(M * N, np.float32))
    diff = np.flatnonzero(C != plain)
    kernels[str(kid)] = {"variant": variant, "M": M, "N": N, "K": K,
                         "sha256": {"A": sha(A), "B": sha(B), "C": sha(C)},
                         "diff_idx": diff.tolist(), "diff_val": [float(x) for x in C[diff]]}
    print(kid, variant, K, len(diff), "elements differ from the oracle product")
checks = {"verify_matrix_160": verify_160, "kernels_cpu": kernels}
(out_dir / "ref_checks.json").write_text(json.dumps(checks, indent=1) + "\n")
