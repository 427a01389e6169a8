"""Host-side logic of the multi-GPU path, on CPU: the P x Q block partition and the verdict all-reduce
(world_size 2, gloo).  The sharded product itself is checked on the CPU with the oracle standing in for each rank's
GPU kernel: stitched blocks == the unsharded product, bit for bit (no collective touches the data path)."""
import os
import socket

import numpy as np
import pytest


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_shard_grid_and_extents(ft):
    from importlib import import_module
    sh = import_module("ftsgemm_b200.sharding")
    assert [sh.shard_grid(w) for w in (1, 2, 4, 8)] == [(1, 1), (1, 2), (2, 2), (2, 4)]  # SURVEY.md 8e
    for world in (1, 2, 4, 8):
        M, N = 32768, 32768
        cover = np.zeros((M // 128, N // 128), np.int32)
        for r in range(world):
            e = sh.shard_extents(r, world, M, N)
            cover[e["m_lo"] // 128:e["m_hi"] // 128, e["n_lo"] // 128:e["n_hi"] // 128] += 1
            assert (e["m_hi"] - e["m_lo"]) * world // e["P"] // e["Q"] > 0
        assert (cover == 1).all()  # every C tile owned exactly once
    # ragged sizes still partition exactly
    e0, e1 = sh.shard_extents(0, 2, 1000, 1000), sh.shard_extents(1, 2, 1000, 1000)
    assert (e0["n_lo"], e0["n_hi"], e1["n_lo"], e1["n_hi"]) == (0, 512, 512, 1000)


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    from importlib import import_module
    from oracle import oracle as O
    ge.load_package()
    sh = import_module("ftsgemm_b200.sharding")
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    M = N = 256
    K = 96
    rng = np.random.default_rng(0)
    A = (rng.integers(-9, 10, M * K) * 0.1).astype(np.float32)
    B = (rng.integers(-9, 10, N * K) * 0.1).astype(np.float32)
    e = sh.shard_extents(rank, world, M, N)
    A2, B2 = O.as2d(A, M, K), O.as2d(B, N, K)
    Ap, Bp = O.colmajor(A2[e["m_lo"]:e["m_hi"]]), O.colmajor(B2[e["n_lo"]:e["n_hi"]])
    mb, nb = e["m_hi"] - e["m_lo"], e["n_hi"] - e["n_lo"]
    Cb = O.sgemm_nt(mb, nb, K, 1.0, Ap, Bp, 0.0, np.zeros(mb * nb, np.float32))  # stand-in for the rank's GPU kernel
    stats = {"tiles": (mb // 128) * (nb // 128), "rows_checked": mb * (nb // 128), "detected": rank, "corrected": rank,
             "uncorrectable": 0, "checksum_faults": 0, "max_abs_residual": 1e-4 * (rank + 1), "max_rel_residual": 1e-7}
    verdict = sh.allreduce_verdict(stats, dist)
    # the per-step device-vector form (CPU tensors + gloo here; ftsgemm_stats_device + NCCL on GPUs)
    vec = [float(stats[k]) for k in sh.STAT_KEYS_SUM] + [float(stats[k]) for k in sh.STAT_KEYS_MAX]
    steps_done = {"n": 0}

    def fill(buf):
        steps_done["n"] += 1
        buf.copy_(torch.tensor(vec, dtype=torch.float64) * torch.tensor([steps_done["n"]] * 6 + [1, 1], dtype=torch.float64))

    ex = sh.VerdictExchange(fill, dist)
    for _ in range(6):  # more steps than slots: slots are recycled
        ex.step()
    v2 = ex.verdict()
    assert v2["rows_checked"] == 6 * verdict["rows_checked"] and v2["detected"] == 6 * verdict["detected"]
    assert abs(v2["max_abs_residual"] - verdict["max_abs_residual"]) < 1e-15 and v2["clean"] == verdict["clean"]
    assert len(v2["per_rank_rows_checked"]) == world
    blocks = [None] * world
    dist.all_gather_object(blocks, (e, Cb))
    if rank == 0:
        full = np.zeros((M, N), np.float32)
        for ee, cb in blocks:
            full[ee["m_lo"]:ee["m_hi"], ee["n_lo"]:ee["n_hi"]] = O.as2d(cb, ee["m_hi"] - ee["m_lo"], ee["n_hi"] - ee["n_lo"])
        want = O.as2d(O.sgemm_nt(M, N, K, 1.0, A, B, 0.0, np.zeros(M * N, np.float32)), M, N)
        q.put((bool(np.array_equal(full, want)), verdict))
    dist.destroy_process_group()


def test_world2_gloo_sharded_product_and_verdict(ft):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ok, verdict = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert ok
    assert verdict["tiles"] == 4 and verdict["detected"] == 1 and verdict["corrected"] == 1 and verdict["clean"]
    assert abs(verdict["max_abs_residual"] - 2e-4) < 1e-12


def _nccl_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    from importlib import import_module
    pkg = ge.load_package()
    sh = import_module("ftsgemm_b200.sharding")
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ft = pkg.FtSgemm()
    n = 1536
    g = torch.Generator(device="cuda").manual_seed(5 + rank)
    dA = torch.randint(-9, 10, (n * n,), generator=g, device="cuda").float() * 0.1
    dB = torch.randint(-9, 10, (n * n,), generator=g, device="cuda").float() * 0.1
    dC = torch.zeros(n * n, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    ex = sh.VerdictExchange(lambda buf: ft.stats_device(buf, stream), dist, dev)
    # rank 1 injects one fault per step: the distributed verdict must show it on every rank
    faults = [{"row": 3, "col": 700, "xor": 1 << 30}] if rank == 1 else None
    for _ in range(5):
        ft.run(31, n, n, n, dA, dB, dC, 1.0, 0.0, pkg.make_opts(stream=stream, faults=faults))
        ex.step()
    v = ex.verdict()
    local = ft.stats()
    # the same exchange FUSED into the kernel: peer stores over NVLink from the last CTA of every launch, no collective
    pv = sh.PeerVerdict(ft, dist)
    n0 = ft.launch_count()
    for _ in range(7):
        ft.run(31, n, n, n, dA, dB, dC, 1.0, 0.0, pkg.make_opts(stream=stream, faults=faults))
    fused_launches = ft.launch_count() - n0
    v2 = pv.verdict()
    local2 = ft.stats()
    q.put((rank, v, local["rows_checked"], v2, local2["rows_checked"], fused_launches))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_world2_nccl_device_verdict_exchange(cuda, ft):
    """The multi-GPU exchange step on real GPUs: two ranks, NCCL all-gather of the device-side verdict vectors."""
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(2)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, v, local_rows, v2, local_rows2, fused_launches in res:
        assert v["detected"] == 5 and v["corrected"] == 5 and v["clean"], v
        assert v["rows_checked"] == 2 * local_rows == 2 * 5 * 1536 * 6
        assert v["per_rank_rows_checked"] == [local_rows, local_rows]
        assert v2["detected"] == 7 and v2["corrected"] == 7 and v2["clean"], v2
        assert v2["rows_checked"] == 2 * local_rows2 == 2 * 7 * 1536 * 6
        assert fused_launches == 7  # one kernel per GEMM, the exchange included
