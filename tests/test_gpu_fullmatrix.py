"""Every element of C against a float64 reference, at the sizes and shapes bench.py times and where a persistent,
planner-driven kernel goes wrong: many waves, cut tiles, carrier tiles, checksum items, wave re-synchronisation,
k-lockstep, ragged edges under the 2-D TMA view, long K, inputs the detection threshold was not calibrated on,
non-finite operands, the beta = 0 / alpha = 0 contract and workspace reuse across calls.

The reference and the comparator are oracle/fullref.py: P = At^T Bt and S = |At|^T |Bt| in float64 (At, Bt = TF32-truncated
operands), ref = alpha * P + beta * C0, and an element passes iff
    |got - ref| <= eps * |alpha| * S + 2^-23 * (|alpha * P| + |beta * C0|),
eps = fullref.eps_for(K, distribution) (measured on a B200 with 4x margin, profiles/r03_fullmatrix_residuals.jsonl).
The comparator is pinned against oracle.sgemm_nt_tf32_model and kept honest by negative controls: on the CPU (a tile that
misses one k-block, a transposed tile, one element 2^10 ulp off) and on the GPU (one 256 x 256 tile of a K - 32 product
spliced into a verified C at 4096^3 and 16384^3): exactly the spliced region is flagged.
"""
import numpy as np
import pytest
import torch

from oracle import fullref as R

SLOW = pytest.mark.slow
GPU = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------- helpers
def _plain_twin(kid):
    return {31: 21, 32: 22}.get(kid, kid - 10)


class _Knobs:
    """ft.debug_set for the duration of a `with` block; every knob back to automatic (-1) afterwards."""

    def __init__(self, ft, **kv):
        self.ft, self.kv = ft, kv

    def __enter__(self):
        try:
            for k, v in self.kv.items():
                self.ft.debug_set(k, v)
        except BaseException:
            self.__exit__()
            raise
        return self

    def __exit__(self, *exc):
        for k in self.kv:
            self.ft.debug_set(k, -1)
        return False


def _operands(M, N, K, dist="ref", seed=0, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    A = R.fill(torch.empty(M * K, device=device), dist, g, M, K)
    B = R.fill(torch.empty(N * K, device=device), dist, g, N, K)
    C0 = torch.randn(M * N, generator=g, device=device)
    return A, B, C0


def _run(h, kid, M, N, K, A, B, C0, alpha=1.0, beta=-1.5, opts=None):
    C = C0.clone()
    h.run(kid, M, N, K, A, B, C, alpha, beta, opts)
    torch.cuda.synchronize()
    return C


def _tile_of(ft, kid):
    return [k for k in ft.kernel_table() if k["id"] == kid][0]["tile"]


def _expect_clean_stats(ft, kid, M, N, st):
    tm, tn = _tile_of(ft, kid)[:2]
    tiles_n = -(-N // tn)
    assert st["detected"] == 0 and st["uncorrectable"] == 0 and st["recomputed"] == 0, (kid, st)
    assert st["tiles"] == (tm // 128) * -(-M // tm) * tiles_n, (kid, M, N, st["tiles"])  # (128-row CTA tiles)
    assert M * tiles_n <= st["rows_checked"] <= tm * -(-M // tm) * tiles_n, (kid, M, N, st["rows_checked"])


def _assert_passes(ref, got, eps, what):
    nbad, where, ratio = ref.check(got, eps)
    print(f"[fullmatrix] {what}: max|got-ref|/(|alpha|S) = {ratio:.3e}  eps = {eps:.3e}  failing = {nbad}")
    assert nbad == 0, (what, nbad, where, ratio, eps)
    return ratio


@pytest.fixture(scope="module")
def h(cuda, ft):
    cuda.cuda.set_device(0)
    x = ft.FtSgemm()
    yield x
    x.close()


@pytest.fixture(scope="module")
def num_sms(cuda):
    return cuda.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(autouse=True)
def _free_cache():
    yield
    if torch.cuda.is_available():
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------- 1. the comparator (CPU)
def test_reference_matches_tf32_model(oracle):
    """The float64 reference equals oracle.sgemm_nt_tf32_model (numpy, float64, rounded to FP32) to FP32 rounding."""
    rng = np.random.default_rng(21)
    M, N, K = 96, 200, 333
    A = rng.standard_normal(M * K).astype(np.float32)
    B = rng.standard_normal(N * K).astype(np.float32)
    C0 = rng.standard_normal(M * N).astype(np.float32)
    model = oracle.sgemm_nt_tf32_model(M, N, K, 0.75, A, B, -1.5, C0, "trunc")
    ref = R.Reference(M, N, K, torch.from_numpy(A), torch.from_numpy(B), torch.from_numpy(C0), 0.75, -1.5,
                      panel_bytes=1 << 16)  # (several panels)
    got = ref.ref.t().numpy().reshape(-1, order="F")  # N x M row-major -> flat column-major
    assert np.all(np.abs(got - model.astype(np.float64)) <= 2.0 ** -24 * np.abs(model) + 1e-30)
    # and the rounded reference passes its own comparator with eps = 0 (only the final-rounding term)
    assert ref.check(torch.from_numpy(model), 0.0)[0] == 0


def _exact_fp32(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    A, B, C0 = (R.fill(torch.empty(M * K), "ref", g), R.fill(torch.empty(N * K), "ref", g), torch.randn(M * N, generator=g))
    ref = R.Reference(M, N, K, A, B, C0, 1.0, -1.5)
    return A, B, C0, ref, ref.ref.float().reshape(-1)  # flat column-major C, the reference rounded to FP32


@pytest.mark.parametrize("K", [256, 4096])
def test_comparator_negative_controls_cpu(K):
    """Splice a wrong region into an otherwise exact FP32 result: the comparator flags elements inside it, none outside."""
    M = N = 512
    A, B, C0, ref, exact = _exact_fp32(M, N, K, K)
    eps = R.eps_for(K)
    assert ref.check(exact, eps)[0] == 0
    n0, m0 = 256, 0  # tile (0, 1): rows 0..255, columns 256..511
    region = torch.zeros(N, M, dtype=torch.bool)
    region[n0:n0 + 256, m0:m0 + 256] = True
    # (a) one k-block (32 k) left out of the tile's product
    At = R.tf32_trunc(A.view(K, M)).double()
    Bt = R.tf32_trunc(B.view(K, N)).double()
    keep = torch.ones(K, dtype=torch.bool)
    keep[64:96] = False
    part = (Bt[keep][:, n0:n0 + 256].t() @ At[keep][:, m0:m0 + 256]) - 1.5 * C0.view(N, M)[n0:n0 + 256, m0:m0 + 256].double()
    # (b) the tile transposed, (c) one element moved by 2^10 ulp
    for what in ("missing k-block", "transposed", "1024 ulp"):
        got = exact.clone().view(N, M)
        if what == "missing k-block":
            got[n0:n0 + 256, m0:m0 + 256] = part.float()
        elif what == "transposed":
            got[n0:n0 + 256, m0:m0 + 256] = got[n0:n0 + 256, m0:m0 + 256].t().clone()
        else:
            r, c = divmod(int(got[n0:n0 + 256, m0:m0 + 256].abs().argmax()), 256)
            got.view(torch.int32)[n0 + r, m0 + c] += 1024
        bad = ref.bad_mask(got.reshape(-1), eps)
        assert not bool((bad & ~region).any()), what
        flagged = int((bad & region).sum())
        assert flagged >= (1 if what == "1024 ulp" else 0.9 * 256 * 256), (what, flagged)


# ---------------------------------------------------------------------------------------------------- 2. the bench sweep
SWEEP = [pytest.param(1024 * i, marks=[GPU, SLOW] if i == 16 else [GPU]) for i in range(1, 17)]


@pytest.mark.parametrize("n", SWEEP)
def test_sweep_whole_matrix(cuda, ft, h, n):
    """bench.py's sweep regime (reference distribution, alpha = 1, beta = -1.5, random C0), every element: the AUTO ids and
    the ids they resolve to bit-equal, ABFT bit-equal to its plain twin, all inside the bound, nothing flagged.  At 4096 and
    16384 the negative control: one tile of a K - 32 product spliced into the verified C is flagged, and only it."""
    M = N = K = n
    A, B, C0 = _operands(M, N, K, "ref", seed=n)
    ref = R.Reference(M, N, K, A, B, C0, 1.0, -1.5)
    eps = R.eps_for(K)
    out = {}
    for auto, is_ft in ((ft.ID_ABFT_AUTO, True), (ft.ID_SGEMM_AUTO, False)):
        kid = ft.select_kernel(M, N, K, is_ft)
        h.stats()
        a = _run(h, auto, M, N, K, A, B, C0)
        st_a = h.stats()
        b = _run(h, kid, M, N, K, A, B, C0)
        st_b = h.stats()
        assert torch.equal(a, b), (n, auto, kid)
        del b
        if is_ft:
            _expect_clean_stats(ft, kid, M, N, st_a)
            _expect_clean_stats(ft, kid, M, N, st_b)
            print(f"[fullmatrix] n={n} id {kid}: max_rel_residual {st_a['max_rel_residual']:.3e}")
        out[is_ft] = (kid, a)
    kid, got = out[True]
    twin = _plain_twin(kid)
    plain = out[False][1] if out[False][0] == twin else _run(h, twin, M, N, K, A, B, C0)
    assert torch.equal(got, plain), (n, kid, twin)
    del out, plain
    _assert_passes(ref, got, eps, f"sweep n={n} id {kid}")
    if n in (4096, 16384):  # negative control: K - 32 on the same pointers (k is the slow index: a prefix)
        short = _run(h, kid, M, N, K - 32, A, B, C0)
        tm, tn = (M // 256) // 2 + 1, (N // 256) - 2
        spliced = got.clone().view(N, M)
        spliced[tn * 256:(tn + 1) * 256, tm * 256:(tm + 1) * 256] = short.view(N, M)[tn * 256:(tn + 1) * 256, tm * 256:(tm + 1) * 256]
        del short
        bad = ref.bad_mask(spliced.view(-1), eps)
        inside = int(bad[tn * 256:(tn + 1) * 256, tm * 256:(tm + 1) * 256].sum())
        total = int(bad.sum())
        print(f"[fullmatrix] negative control n={n}: tile (m {tm}, n {tn}) of a K-32 product spliced in: "
              f"{inside} of 65536 elements flagged inside, {total - inside} outside")
        assert total == inside and inside >= 0.9 * 65536, (n, inside, total)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096, 8192])
@pytest.mark.parametrize("kid", [16, 15])
def test_literal_tiles_whole_matrix(cuda, ft, h, n, kid):
    """The 128-row tiles of the reference's table (huge 128 x 128, wide 128 x 256) at full size, every element."""
    M = N = K = n
    A, B, C0 = _operands(M, N, K, "ref", seed=n + kid)
    ref = R.Reference(M, N, K, A, B, C0, 1.0, -1.5)
    plain = _run(h, _plain_twin(kid), M, N, K, A, B, C0)
    h.stats()
    got = _run(h, kid, M, N, K, A, B, C0)
    _expect_clean_stats(ft, kid, M, N, h.stats())
    assert torch.equal(got, plain)
    del plain
    _assert_passes(ref, got, R.eps_for(K), f"n={n} id {kid}")


# ---------------------------------------------------------------------------------------------------- 3. ragged / multi-wave / extreme
def _sched_facts(ft, kid, M, N, K, num_sms):
    hdr, segs = ft.debug_schedule(kid, M, N, K, num_sms)
    data = [s for s in segs if not s["is_chk"]]
    return hdr, segs, {
        "carriers": sum(1 for s in data if s["kind"] == 6),
        "cut": hdr["sk_tiles"],
        "chk_items": hdr["n_chk_tiles"],
        "data_tiles": hdr["num_tiles"] - hdr["n_chk_tiles"],
        "chk_slices": hdr["chk_slices"],
        "waves": (hdr["num_tiles"] - hdr["n_chk_tiles"]) / hdr["units"],  # data tiles per unit
        "all_waves": hdr["num_tiles"] / hdr["units"],
        "lockstep": 4.0 * K * (M + N) > 96 * 2 ** 20,
    }


RAGGED = [
    # (M, N, K), ABFT id, what must be in the plan
    ((4100, 4196, 4127), 31, lambda f: f["cut"] > 0 and f["chk_items"] > 0 and f["waves"] > 3.5),
    ((4096, 4064, 4096), 31, lambda f: f["carriers"] > 0 and f["chk_items"] == 0 and f["cut"] > 0),
    ((4096, 4100, 4096), 31, lambda f: f["carriers"] == 0 and f["chk_items"] > 0),
    ((3072, 3072, 3072), 31, lambda f: f["chk_items"] > 0 and f["waves"] < 2.0 < f["all_waves"] < 3.0),
    ((2052, 12288, 1000), 31, lambda f: f["chk_items"] > 0 and f["waves"] > 5),
    ((12288, 2052, 1000), 31, lambda f: f["chk_items"] > 0 and f["cut"] > 0),
    ((6144, 6144, 12288), 31, lambda f: f["lockstep"] and f["cut"] > 0),
    ((12292, 12292, 1100), 31, lambda f: f["lockstep"] and f["waves"] >= 24 and f["cut"] > 0),
    ((256, 65536, 1024), 31, lambda f: f["chk_items"] == 4 and f["data_tiles"] == 256),
    ((65536, 256, 1024), 31, lambda f: f["carriers"] == 0 and f["chk_items"] == 256 and f["data_tiles"] == 256),
    ((1024, 1024, 65536), 32, lambda f: f["chk_slices"] > 1),
]


def _fault_sites(ft, kid, M, N, K, num_sms, rng):
    """Up to 8 faults at positions the schedule makes interesting, never two in one (row, tile) and never two in one row."""
    BM, BN = _tile_of(ft, kid)[:2]
    _, segs, _ = _sched_facts(ft, kid, M, N, K, num_sms)
    data = [s for s in segs if not s["is_chk"]]
    sites = [(0, 0), (M - 1, N - 1), (max(0, M - 1 - 37), max(0, N - 1 - 100))]
    for kind in (6, 2):
        s = next((s for s in data if s["kind"] == kind), None)
        if s is not None:
            sites.append((min(M - 1, s["m_blk"] * BM + 130), min(N - 1, s["n_blk"] * BN + 77)))
    # one per checksum group (the data tile-columns whose checksums one checksum tile-column holds: BN / 4 of them)
    tiles_n = -(-N // BN)
    for g0 in range(0, tiles_n, BN // 4):
        if len(sites) >= ft.MAX_FAULTS:
            break
        tn = min(tiles_n - 1, g0 + int(rng.integers(0, BN // 4)))
        sites.append((int(rng.integers(0, M)), min(N - 1, tn * BN + int(rng.integers(0, BN)))))
    out, rows = [], set()
    for r, c in sites:
        if r in rows:
            continue
        rows.add(r)
        out.append((r, c))
    return out[:ft.MAX_FAULTS]


@pytest.mark.parametrize("shape,kid,plan", [pytest.param(*x, marks=[GPU, SLOW] if x[0][2] == 65536 else [GPU]) for x in RAGGED],
                         ids=[f"{s[0]}x{s[1]}x{s[2]}" for s, _, _ in RAGGED])
def test_ragged_multiwave_extreme(cuda, ft, h, num_sms, shape, kid, plan):
    M, N, K = shape
    _, _, facts = _sched_facts(ft, kid, M, N, K, num_sms)
    assert plan(facts), (shape, facts)  # the planner path this shape exists for really occurs
    A, B, C0 = _operands(M, N, K, "ref", seed=M * 7 + N * 3 + K)
    ref = R.Reference(M, N, K, A, B, C0, 1.0, -1.5)
    plain = _run(h, _plain_twin(kid), M, N, K, A, B, C0)
    h.stats()
    got = _run(h, kid, M, N, K, A, B, C0)
    _expect_clean_stats(ft, kid, M, N, h.stats())
    assert torch.equal(got, plain), shape
    del plain
    _assert_passes(ref, got, R.eps_for(K), f"{shape} id {kid}")
    # carriers forced on / off where the shape allows them: the same C
    if shape in ((4096, 4064, 4096), (4096, 4100, 4096)):
        for carriers in (0, 1):
            with _Knobs(ft, carriers=carriers):
                assert torch.equal(_run(h, kid, M, N, K, A, B, C0), got), (shape, carriers)
    # three runs with every whole tile cut into 3 pieces: the park / seed chain gives the same bits every time
    with _Knobs(ft, splitk=3):
        for rep in range(3):
            assert torch.equal(_run(h, kid, M, N, K, A, B, C0), got), (shape, rep)
    assert h.stats()["detected"] == 0
    # faults at the interesting places: all corrected in place, nothing else changes
    rng = np.random.default_rng(M + N + K)
    sites = _fault_sites(ft, kid, M, N, K, num_sms, rng)
    faults = [{"row": r, "col": c, **({"xor": 1 << 30} if i % 2 else {"add": 1000.0})} for i, (r, c) in enumerate(sites)]
    fixed = _run(h, kid, M, N, K, A, B, C0, opts=ft.make_opts(faults=faults))
    st = h.stats()
    assert st["detected"] == len(faults) and st["uncorrectable"] == 0, (shape, faults, st)
    assert st["corrected"] + st["recomputed"] == len(faults), (shape, faults, st)
    if K <= 8192:  # (beyond, tau_rel grows with K and a flip that leaves a small upset is detected but not located)
        assert st["corrected"] == len(faults), (shape, faults, st)
    redo = {e["row"] for e in st["events"] if e["status"] == 5}  # a recomputed row segment is re-rounded as a whole
    diff = (fixed != got).view(N, M).nonzero().tolist()
    assert all((m, n) in sites or m in redo for n, m in diff), (shape, diff[:10], redo)
    _assert_passes(ref, fixed, R.eps_for(K), f"{shape} id {kid} with {len(faults)} corrected faults")


# ---------------------------------------------------------------------------------------------------- 4. uncalibrated inputs
DISTS = ["ref", "normal", "uniform01", "wide"]
CASES = [((2048, 2048, 2048), 31), ((2048, 2048, 2048), 16), ((4096, 4096, 4096), 31), ((4096, 4096, 4096), 16),
         ((1024, 1024, 16384), 31), ((1024, 1024, 32768), 31), ((1024, 1024, 65536), 31)]


@pytest.mark.parametrize("dist", DISTS)
@pytest.mark.parametrize("shape,kid", [pytest.param(s, k, marks=[GPU, SLOW] if s[2] == 65536 else [GPU]) for s, k in CASES],
                         ids=[f"{s[0]}x{s[1]}x{s[2]}-id{k}" for s, k in CASES])
def test_threshold_on_uncalibrated_inputs(cuda, ft, h, shape, kid, dist):
    """Fault-free runs on distributions the threshold was not calibrated on (non-negative operands, 2^+-20 dynamic range),
    and at long K: nothing flagged, ABFT bit-equal to plain, every element inside the bound."""
    M, N, K = shape
    A, B, C0 = _operands(M, N, K, dist, seed=K + kid + DISTS.index(dist))
    ref = R.Reference(M, N, K, A, B, C0, 1.0, -1.5)
    plain = _run(h, _plain_twin(kid), M, N, K, A, B, C0)
    h.stats()
    got = _run(h, kid, M, N, K, A, B, C0)
    st = h.stats()
    print(f"[fullmatrix] {dist} {shape} id {kid}: max_rel_residual {st['max_rel_residual']:.3e} detected {st['detected']}")
    _expect_clean_stats(ft, kid, M, N, st)
    assert torch.equal(got, plain), (shape, kid, dist)
    del plain
    _assert_passes(ref, got, R.eps_for(K, dist), f"{dist} {shape} id {kid}")


# ---------------------------------------------------------------------------------------------------- 5. non-finite operands, beta = 0, alpha = 0
@pytest.mark.gpu
@pytest.mark.parametrize("kid", [31, 16, 15])
def test_nonfinite_operands(cuda, ft, h, kid):
    """+Inf at A[m1, k1], NaN at B[n2, k2], -Inf at A[m3, k3] where column k3 of B is zero (Inf * 0): the ABFT kernel
    stores what the plain kernel stores -- finite elements bit-equal, non-finite ones in the same places -- and does not
    turn a legitimately non-finite element into a finite one."""
    M, N, K = 1024, 1280, 768
    A, B, C0 = _operands(M, N, K, "ref", seed=55)
    (m1, k1), (n2, k2), (m3, k3) = (100, 7), (700, 300), (900, 500)
    B.view(K, N)[k3] = 0.0
    Az, Bz = A.clone(), B.clone()
    A.view(K, M)[k1, m1] = float("inf")
    B.view(K, N)[k2, n2] = float("nan")
    A.view(K, M)[k3, m3] = float("-inf")
    plain = _run(h, _plain_twin(kid), M, N, K, A, B, C0)
    h.stats()
    got = _run(h, kid, M, N, K, A, B, C0)
    st = h.stats()
    print(f"[fullmatrix] non-finite operands id {kid}: {st}")
    fin = torch.isfinite(plain)
    assert torch.equal(fin, torch.isfinite(got)) and torch.equal(torch.isnan(plain), torch.isnan(got))
    assert torch.equal(got[fin], plain[fin])
    assert torch.equal(got[~fin & ~torch.isnan(got)], plain[~fin & ~torch.isnan(plain)])  # same infinities
    Cg = got.view(N, M)
    assert not bool(torch.isfinite(Cg[:, m1]).any()) and not bool(torch.isfinite(Cg[:, m3]).any())
    assert not bool(torch.isfinite(Cg[n2]).any())
    assert st["uncorrectable"] == 0
    # everything outside rows m1, m3 and column n2 is finite and inside the bound of the product without those entries
    ref = R.Reference(M, N, K, Az, Bz, C0, 1.0, -1.5)
    bad = ref.bad_mask(got, R.eps_for(K))
    bad[:, [m1, m3]] = False
    bad[n2] = False
    assert int(bad.sum()) == 0


_BETA0_OPTS = [("default", {}), ("precision=1", {"precision": 1}), ("check_segments=3", {"check_segments": 3}),
               ("protect_epilogue", {"protect_epilogue": True})]


@pytest.mark.gpu
def test_beta_zero_never_reads_c_and_alpha_zero_keeps_c(cuda, ft, h):
    """BLAS: beta = 0 means C is not read -- a C full of NaN gives what C = 0 gives (every id, the AUTO ids, 3xTF32, intra-K
    checking, the protected epilogue, the host-buffer path with 3 column panels); alpha = 0, beta = 1 leaves C unchanged."""
    M, N, K = 512, 1000, 320  # N ragged for every tile width: the ragged store path as well
    A, B, _ = _operands(M, N, K, "ref", seed=9)
    zeros = torch.zeros(M * N, device="cuda")
    nans = torch.full((M * N,), float("nan"), device="cuda")
    C1 = torch.randn(M * N, device="cuda")
    ids = sorted({k["id"] for k in ft.kernel_table()} | {ft.ID_SGEMM_AUTO, ft.ID_ABFT_AUTO})
    ft_ids = {k["id"] for k in ft.kernel_table() if k["fault_tolerant"]} | {ft.ID_ABFT_AUTO}
    for kid in ids:
        variants = _BETA0_OPTS if kid in (31, 16) else _BETA0_OPTS[:1]
        for name, kw in variants:
            want = _run(h, kid, M, N, K, A, B, zeros, 0.75, 0.0, ft.make_opts(**kw))
            got = _run(h, kid, M, N, K, A, B, nans, 0.75, 0.0, ft.make_opts(**kw))
            assert torch.equal(got, want), (kid, name, int(torch.isnan(got).sum()))
        h.stats()
        same = _run(h, kid, M, N, K, A, B, C1, 0.0, 1.0)
        st = h.stats()
        assert torch.equal(same, C1), (kid, "alpha = 0")
        if kid in ft_ids:
            assert st["detected"] == 0, (kid, st)
    hA, hB = A.cpu().numpy(), B.cpu().numpy()
    with _Knobs(ft, host_panels=3):
        for kid in (31, 16):
            want = _run(h, kid, M, N, K, A, B, zeros, 0.75, 0.0).cpu().numpy()
            hC = np.full(M * N, np.nan, np.float32)
            h.run_host(kid, M, N, K, hA, hB, hC, 0.75, 0.0, None)
            assert np.array_equal(hC, want), kid
    assert h.stats()["detected"] == 0


# ---------------------------------------------------------------------------------------------------- 6. stale workspace
@pytest.mark.gpu
def test_workspace_reuse_matches_fresh_handle(cuda, ft, h):
    """A seeded sequence of ~20 calls on one handle (shapes growing and shrinking, FT and plain ids, checksum K-slices
    1 <-> 4, cached checksum vectors, 3xTF32, intra-K checking): every result bit-equal to the same call on a fresh handle."""
    shapes = [(1024, 1024, 1024), (4096, 4100, 2048), (512, 768, 640), (2048, 2048, 4096), (260, 388, 72), (3072, 1024, 1536)]
    ops = {s: _operands(*s, "ref", seed=i) for i, s in enumerate(shapes)}
    rng = np.random.default_rng(2024)
    seq = []
    while len(seq) < 20:
        s = shapes[int(rng.integers(len(shapes)))]
        kid = int(rng.choice([31, 21, 16, 6, 32, 40, 20]))
        kw = {}
        r = rng.random()
        if r < 0.15 and kid in (31, 16, 32, 40):
            kw = {"precision": 1}
        elif r < 0.3 and kid in (31, 16, 32, 40):
            kw = {"check_segments": 3}
        seq.append((s, kid, kw, False, int(rng.choice([1, 4]))))
        if rng.random() < 0.3:  # the same call twice more: the second one reuses the checksum vectors of B (unchanged)
            seq.append((s, kid, {}, False, seq[-1][4]))
            seq.append((s, kid, {}, kid in (31, 16, 32, 40), seq[-1][4]))
    outs = []
    for s, kid, kw, reuse, slices in seq:
        A, B, C0 = ops[s]
        with _Knobs(ft, chk_slices=slices):
            outs.append(_run(h, kid, *s, A, B, C0, 0.75, -1.5, ft.make_opts(reuse_b_checksums=reuse, **kw)).cpu())
    assert h.stats()["detected"] == 0
    for (s, kid, kw, reuse, slices), got in zip(seq, outs):
        A, B, C0 = ops[s]
        fresh = ft.FtSgemm()
        try:
            with _Knobs(ft, chk_slices=slices):
                want = _run(fresh, kid, *s, A, B, C0, 0.75, -1.5, ft.make_opts(**kw)).cpu()
            assert fresh.stats()["detected"] == 0
        finally:
            fresh.close()
        assert torch.equal(got, want), (s, kid, kw, reuse, slices)
