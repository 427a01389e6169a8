"""Float64 reference of a whole C = alpha * A * B^T + beta * C0 and an element-wise comparator, computed with torch on
whatever device the operands live on (on the GPU this is a float64 GEMM of the vendor library, independent of the
kernels under test).

Layout as in include/ftsgemm.h: A is M x K, B is N x K, C is M x N, all column-major, so A.view(K, M), B.view(K, N) and
C.view(N, M) are row-major views with k (resp. n) the slow index.

With single-pass TF32 (opts.precision = 0) the tensor core reads A and B with the 13 low mantissa bits cleared; the
reference uses those operands (At, Bt):

    P = At^T Bt,   S = |At|^T |Bt|   (float64),   ref = alpha * P + beta * C0,

and an element passes iff

    |got - ref| <= eps * |alpha| * S + 2^-23 * (|alpha * P| + |beta * C0|).

eps covers the FP32 accumulation of the K products; the second term the final FP32 alpha * acc + beta * c.  For
opts.precision = 1 (3xTF32) the operands are not truncated.  The rule for eps is eps_for() below.
"""
from __future__ import annotations

import math

import torch

U23 = 2.0 ** -23


def tf32_trunc(t: torch.Tensor) -> torch.Tensor:
    """FP32 values with the 13 low mantissa bits cleared (what kind::tf32 reads; as oracle.tf32_trunc)."""
    return (t.view(torch.int32) & -8192).view(torch.float32)


def eps_for(K: int, dist: str = "ref") -> float:
    """Accumulation allowance eps as a fraction of S for an inner dimension K.

    Zero-mean operands ("ref", "normal", "wide"): the rounding errors of the FP32 accumulator cancel like a random walk,
    eps = EPS_ZERO_MEAN * sqrt(K / 1024).  Non-negative operands ("uniform01"): every partial sum grows with k and the
    accumulator's truncation-like rounding adds up linearly, eps = EPS_NONNEG * K / 1024.  The constants are 4x the
    largest ratio max(|got - ref| - rounding term) / (|alpha| * S) measured on a B200 over the cases of
    scripts/fullmatrix_residuals.py (profiles/r03_fullmatrix_residuals.jsonl), scaled to K = 1024 by the same law:
    zero-mean 7.5e-7 (N(0,1), 4096^3; the reference distribution gives 6.3e-7 .. 7.0e-7 from 1024^3 to 16384^3),
    U[0,1) 7.5e-6 (2048^3 and 4096^3: 1.5e-5 and 3.0e-5)."""
    if dist == "uniform01":
        return EPS_NONNEG * K / 1024.0
    return EPS_ZERO_MEAN * math.sqrt(K / 1024.0)


EPS_ZERO_MEAN = 3e-6
EPS_NONNEG = 3e-5


class Reference:
    """ref (float64), S and the rounding term (float32), all N x M (the transposed, row-major view of column-major C).
    Built in panels of C's columns so that the float64 temporaries stay within `panel_bytes`."""

    def __init__(self, M, N, K, A, B, C0, alpha, beta, precision=0, panel_bytes=1 << 30):
        self.M, self.N, self.K, self.alpha, self.beta = M, N, K, float(alpha), float(beta)
        At, Bt = A.view(K, M), B.view(K, N)
        if precision == 0:
            At, Bt = tf32_trunc(At), tf32_trunc(Bt)
        dev = A.device
        self.ref = torch.empty(N, M, dtype=torch.float64, device=dev)
        self.S = torch.empty(N, M, dtype=torch.float32, device=dev)
        self.fp = torch.empty(N, M, dtype=torch.float32, device=dev)
        A64 = At.double()
        Aabs = A64.abs()
        C0t = C0.view(N, M) if (C0 is not None and beta != 0.0) else None
        w = max(1, min(N, panel_bytes // (8 * (M + K) * 3)))
        for j0 in range(0, N, w):
            j1 = min(N, j0 + w)
            Bp = Bt[:, j0:j1].double()                   # K x w
            P = Bp.t() @ A64                             # w x M
            self.S[j0:j1] = (Bp.abs_().t() @ Aabs).float()
            del Bp
            P.mul_(self.alpha)
            fp = P.abs()
            if C0t is not None:
                c = C0t[j0:j1].double().mul_(self.beta)
                P.add_(c)
                fp.add_(c.abs_())
                del c
            self.ref[j0:j1] = P
            self.fp[j0:j1] = fp.mul_(U23).float()
            del P, fp
        del A64, Aabs

    def _err(self, got, j0, j1):
        return (got.view(self.N, self.M)[j0:j1].double() - self.ref[j0:j1]).abs_()

    def _panels(self, rows=1 << 25):
        w = max(1, rows // self.M)
        return [(j0, min(self.N, j0 + w)) for j0 in range(0, self.N, w)]

    def max_ratio(self, got) -> float:
        """max (|got - ref| - rounding term) / (|alpha| * S) over the elements with S > 0: the smallest eps with which got
        passes (the number eps is calibrated on)."""
        worst = 0.0
        for j0, j1 in self._panels():
            d = self._err(got, j0, j1).sub_(self.fp[j0:j1].double()).clamp_min_(0.0)
            s = self.S[j0:j1].double().mul_(abs(self.alpha))
            r = torch.where(s > 0, d / s.clamp_min(1e-300), torch.zeros_like(d))
            worst = max(worst, float(r.max()))
        return worst

    def bad_mask(self, got, eps) -> torch.Tensor:
        """Boolean N x M mask of the elements outside the bound (NaN / Inf in got are outside)."""
        out = torch.empty(self.N, self.M, dtype=torch.bool, device=self.ref.device)
        for j0, j1 in self._panels():
            d = self._err(got, j0, j1)
            tol = self.S[j0:j1].double().mul_(eps * abs(self.alpha)).add_(self.fp[j0:j1].double())
            out[j0:j1] = ~(d <= tol)
        return out

    def check(self, got, eps):
        """(number of failing elements, first few failing (m, n), max ratio)."""
        bad = self.bad_mask(got, eps)
        nbad = int(bad.sum())
        where = [(int(m), int(n)) for n, m in bad.nonzero()[:5].tolist()] if nbad else []
        return nbad, where, self.max_ratio(got)


# ---------------------------------------------------------------------------------------------------- input distributions
def fill(t: torch.Tensor, dist: str, gen: torch.Generator, rows: int = 0, cols: int = 0) -> torch.Tensor:
    """Fill a flat float32 tensor in place.  ref: the reference generator's distribution (magnitude (rand() % 10) * 0.1,
    random sign, utils/utils.cu:23-31, as bench.fill_ref_dist); normal: N(0, 1); uniform01: U[0, 1); wide: N(0, 1)
    with each row of the rows x cols column-major operand scaled by 2^U(-20, 20) (for A and B: rows of A, columns of B^T)."""
    n = t.numel()
    step = 1 << 26
    for i in range(0, n, step):
        v = t[i:i + step]
        if dist == "ref":
            v.copy_(torch.randint(0, 10, (v.numel(),), generator=gen, device=t.device, dtype=torch.int32))
            v.mul_(0.1)
            sgn = torch.randint(0, 2, (v.numel(),), generator=gen, device=t.device, dtype=torch.int32)
            v.mul_(sgn.float().mul_(2).sub_(1))
        elif dist in ("normal", "wide"):
            v.normal_(generator=gen)
        elif dist == "uniform01":
            v.uniform_(0.0, 1.0, generator=gen)
        else:
            raise ValueError(dist)
    if dist == "wide":
        e = torch.randint(-20, 21, (rows,), generator=gen, device=t.device).float()
        t.view(cols, rows).mul_(torch.exp2(e))
    return t
