"""
Row-parallel GEMM with the tensor-parallel sum fused into its epilogue (csrc/gemm_tc_i8_ar.cu, exl3b_gemm_allreduce).

CPU part (always runs): eligibility rules, argument validation, the host-side selection in tp.row_parallel_forward.

GPU part (verified on a B200 in round 2, gpurun_out/r02_call1): world-1 equality with the plain kernel and the loop-back
protocol test run on one GPU (-m gpu); the two-process test needs two GPUs and carries the `multigpu` marker instead
(gpurun --gpus 2 -- python -m pytest tests -m multigpu).
"""
import ctypes, os
import numpy as np
import pytest
import torch
from oracle import exl3_oracle as orc



# ---------------------------------------------------------------------------------------------------------------------
# CPU: host logic
# ---------------------------------------------------------------------------------------------------------------------

def test_allreduce_eligibility_rules():
    from exllamav3_b200 import ext
    ok = lambda *a: ext.lib.exl3b_gemm_allreduce_check(*a) == 0
    #          m  k     n     K  cb world max_elems
    assert ok(1, 1024, 4096, 4, 2, 4, 65536)
    assert ok(4, 128, 128, 8, 2, 8, 512)
    assert not ok(5, 1024, 4096, 4, 2, 4, 65536) and b"m <= 4" in ext.lib.exl3b_last_error()
    assert not ok(1, 1024, 4096, 4, 0, 4, 65536) and b"mul1" in ext.lib.exl3b_last_error()
    assert not ok(1, 1024, 4096, 4, 1, 4, 65536)
    assert not ok(1, 1000, 4096, 4, 2, 4, 65536) and b"multiples of 128" in ext.lib.exl3b_last_error()
    assert not ok(1, 1024, 4096, 4, 2, 9, 65536) and b"world size" in ext.lib.exl3b_last_error()
    assert not ok(4, 1024, 4096, 4, 2, 4, 8192) and b"exchange slot" in ext.lib.exl3b_last_error()
    assert ext.exl3_gemm_allreduce_supported(2, 3584, 4096, 4, False, True, 4, 65536)
    assert not ext.exl3_gemm_allreduce_supported(2, 3584, 4096, 4, True, False, 4, 65536)


def test_tp_setup_validation_without_gpu():
    from exllamav3_b200 import ext
    lib = ext.lib
    buf = ctypes.create_string_buffer(64)
    assert lib.exl3b_tp_alloc(0, 9, 1024, ctypes.cast(buf, ctypes.c_void_p)) == -2 and b"world size" in lib.exl3b_last_error()
    assert lib.exl3b_tp_alloc(3, 2, 1024, ctypes.cast(buf, ctypes.c_void_p)) == -2 and b"rank" in lib.exl3b_last_error()
    assert lib.exl3b_tp_alloc(0, 2, 100, ctypes.cast(buf, ctypes.c_void_p)) == -2 and b"max_elems" in lib.exl3b_last_error()
    # argument checks of the fused GEMM fire before any CUDA work
    one = ctypes.c_void_p(16)
    assert lib.exl3b_gemm_allreduce(None, one, one, one, one, None, one, 1, 128, 64, 4, 2, 1) == -1
    assert lib.exl3b_gemm_allreduce(None, one, one, one, one, None, one, 1, 128, 128, 9, 2, 1) == -2
    with pytest.raises(RuntimeError, match="handle bytes"):
        ext.tp_attach(b"x" * 10, 2)
    if not torch.cuda.is_available():
        # no device: the library reports a CUDA error, it does not fall back to anything
        assert lib.exl3b_tp_alloc(0, 2, 1024, ctypes.cast(buf, ctypes.c_void_p)) == -3


def test_row_parallel_forward_selection_host_logic():
    """tp.row_parallel_forward takes the one-kernel path only when enabled and eligible (mul1, <= 4 rows, no bias)."""
    from exllamav3_b200 import tp, QLinear
    k, n, K = 256, 384, 4
    tr, suh, svh, _ = orc.make_synthetic(k, n, K)
    mk = lambda **kw: QLinear(torch.from_numpy(tr), torch.from_numpy(suh), torch.from_numpy(svh), **kw)
    mul1 = mk(mul1=True)
    three = mk()
    biased = mk(mul1=True, bias=torch.zeros(n, dtype=torch.half))
    assert not tp.fused_allreduce_eligible(mul1, 1)                       # not enabled
    saved = dict(tp._fused)
    try:
        tp._fused.update(on=True, world=2, max_elems=4 * 384)
        assert tp.fused_allreduce_eligible(mul1, 1) and tp.fused_allreduce_eligible(mul1, 4)
        assert not tp.fused_allreduce_eligible(mul1, 5)                   # rows
        assert not tp.fused_allreduce_eligible(three, 1)                  # codebook
        assert not tp.fused_allreduce_eligible(biased, 1)                 # bias on this shard
        # rank invariance: the row shard that does NOT hold the bias (first != 0) must give the same answer as the one that does
        s0, s1 = tp.tp_slice(biased, (False, 0, 128)), tp.tp_slice(biased, (False, 128, 256))
        assert s0.bias is not None and s1.bias is None and s0.bias_in_group and s1.bias_in_group
        assert not tp.fused_allreduce_eligible(s0, 1) and not tp.fused_allreduce_eligible(s1, 1)
        u0, u1 = tp.tp_slice(mul1, (False, 0, 128)), tp.tp_slice(mul1, (False, 128, 256))
        assert tp.fused_allreduce_eligible(u0, 1) and tp.fused_allreduce_eligible(u1, 1)
        assert not tp.fused_allreduce_eligible(mul1, 1, any_bias=True)    # bias on some other rank's shard
        tp._fused.update(max_elems=384)
        assert tp.fused_allreduce_eligible(mul1, 1) and not tp.fused_allreduce_eligible(mul1, 2)   # slot size
    finally:
        tp._fused.clear(); tp._fused.update(saved)


# ---------------------------------------------------------------------------------------------------------------------
# GPU (opt-in until verified)
# ---------------------------------------------------------------------------------------------------------------------

def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _plain_gemm(ext, dev, x, tr, suh, svh, K, fp32=True):
    m, n = x.shape[0], tr.shape[1] * 16
    C = torch.empty((m, n), dtype=torch.float if fp32 else torch.half, device=dev)
    tag = ext.exl3_gemm(T(x, dev), T(tr, dev), C, T(suh, dev), torch.empty((m, x.shape[1]), dtype=torch.half, device=dev),
                        T(svh, dev), -1, False, True, 0)
    assert tag == ext.EXL3B_TAG_TC_I8
    return C


@pytest.mark.gpu
@pytest.mark.parametrize("K,m", [(4, 1), (4, 4), (2, 3), (6, 1)])
def test_fused_allreduce_world1_equals_plain_gemm(cuda, K, m):
    """world = 1: no peers; the fused kernel must reproduce exl3_gemm bit for bit (fp32 C) and advance the epoch."""
    from exllamav3_b200 import ext
    k, n = 1024, 2048
    tr, suh, svh, x = orc.make_synthetic(k, n, K, m=m)
    ref = _plain_gemm(ext, cuda, x, tr, suh, svh, K)
    ext.tp_alloc(0, 1, m * n)
    try:
        ext.tp_attach(b"\0" * 64, 1)
        e0 = int(ext.lib.exl3b_tp_debug_epoch())
        for rep in range(3):
            C = torch.full((m, n), float("nan"), dtype=torch.float, device=cuda)
            tag = ext.exl3_gemm_allreduce(T(x, cuda), T(tr, cuda), C, T(suh, cuda), None, T(svh, cuda), False, True)
            assert tag == ext.EXL3B_TAG_TC_I8_AR
            torch.cuda.synchronize()
            assert torch.equal(C, ref)
        assert int(ext.lib.exl3b_tp_debug_epoch()) == e0 + 3
    finally:
        ext.tp_free()


@pytest.mark.gpu
@pytest.mark.parametrize("world,rank", [(2, 0), (2, 1), (4, 2), (8, 7)])
def test_fused_allreduce_loopback_protocol(cuda, world, rank):
    """
    One GPU plays rank `rank` of `world`: the peers' partials (plain exl3_gemm of their row shards) are injected into the
    receive buffer, the fused kernel must (1) return the rank-ordered fp32 sum, (2) have stored its own partial into slot
    [rank] of every peer buffer, (3) have put the sentinel back into its own buffer, (4) alternate slots over launches.
    """
    from exllamav3_b200 import ext
    K, m, k_full, n = 4, 2, 128 * 2 * world, 1024
    tr, suh, svh, x = orc.make_synthetic(k_full, n, K, m=m)
    ks = k_full // world
    parts = []
    for r in range(world):
        sl = slice(r * ks, (r + 1) * ks)
        parts.append(_plain_gemm(ext, cuda, np.ascontiguousarray(x[:, sl]), np.ascontiguousarray(tr[r * ks // 16:(r + 1) * ks // 16]),
                                 suh[sl], svh, K))
    want = torch.zeros_like(parts[0])
    for r in range(world):
        want = want + parts[r]                    # rank order, fp32: exactly the kernel's summation order
    ext.tp_alloc(rank, world, m * n)
    try:
        ext.tp_attach_loopback()
        sl = slice(rank * ks, (rank + 1) * ks)
        xs, trs = T(np.ascontiguousarray(x[:, sl]), cuda), T(np.ascontiguousarray(tr[rank * ks // 16:(rank + 1) * ks // 16]), cuda)
        stream = torch.cuda.current_stream(cuda).cuda_stream
        for rep in range(3):
            e = int(ext.lib.exl3b_tp_debug_epoch())
            for r in range(world):
                if r != rank:
                    assert ext.lib.exl3b_tp_debug_inject(stream, r, parts[r].data_ptr(), m * n) == 0
            C = torch.full((m, n), float("nan"), dtype=torch.float, device=cuda)
            ext.exl3_gemm_allreduce(xs, trs, C, T(suh[sl], cuda), None, T(svh, cuda), False, True)
            torch.cuda.synchronize()
            assert torch.equal(C, want)
            assert int(ext.lib.exl3b_tp_debug_epoch()) == e + 1
            host = np.empty(m * n, dtype=np.uint32)
            for r in range(world):
                if r == rank:
                    continue
                # (2) own partial landed in peer r's buffer, slot e % 2, source = rank
                assert ext.lib.exl3b_tp_debug_peek(r, e % 2, rank, host.ctypes.data, m * n) == 0
                assert (host.view(np.float32).reshape(m, n) == parts[rank].cpu().numpy()).all()
                # (3) own buffer re-armed
                assert ext.lib.exl3b_tp_debug_peek(rank, e % 2, r, host.ctypes.data, m * n) == 0
                assert (host == 0xffffffff).all()
    finally:
        ext.tp_free()


def _two_rank_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from exllamav3_b200 import ext, tp, QLinear
        K, m, k_full, n = 4, 1, 4096, 4096
        tr, suh, svh, x = orc.make_synthetic(k_full, n, K, m=m)
        lin = QLinear(torch.from_numpy(tr), torch.from_numpy(suh), torch.from_numpy(svh), mul1=True, out_dtype=torch.float)
        shard = tp.row_shard(lin, rank, world, dev)
        first, last = tp.split_ranges(k_full, world)[rank]
        xl = torch.from_numpy(np.ascontiguousarray(x[:, first:last])).to(dev)
        y_nccl = tp.row_parallel_forward(shard, xl, {}, torch.float)          # exl3_gemm + NCCL all-reduce
        tp.enable_fused_allreduce(max_elems=4 * n)
        ys = []
        for _ in range(20):                                                     # back to back: slots alternate, peers run ahead
            ys.append(tp.row_parallel_forward(shard, xl, {}, torch.float))
        torch.cuda.synchronize()
        ref = orc.exl3_gemm_f64(x, tr, suh, svh, K, 2)
        err = float(np.abs(ys[-1].cpu().numpy() - ref).max() / np.abs(ref).max())
        same = all(torch.equal(ys[0], y) for y in ys)
        gathered = [torch.empty_like(ys[0]) for _ in range(world)]
        dist.all_gather(gathered, ys[0])
        ident = all(torch.equal(gathered[0], g) for g in gathered)              # rank-ordered sums: bit-identical everywhere
        close = float((ys[0] - y_nccl).abs().max() / y_nccl.abs().max())
        tp.disable_fused_allreduce()
        q.put((rank, err, same, ident, close))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.multigpu
def test_fused_allreduce_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, 29731, q)) for r in range(2)]
    for p in procs: p.start()
    for p in procs: p.join(300)
    res = sorted(q.get(timeout=5) for _ in range(2))
    for rank, err, same, ident, close in res:
        assert err < 2e-3, f"rank {rank}: rel err vs fp64 oracle {err}"
        assert same and ident
        assert close < 1e-5
