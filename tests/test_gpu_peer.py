"""Peer-memory data parallel (thinkdiff_mlre_b200/peer.py): the gradient exchange fused into the weight-gradient GEMM epilogues.

The kernels take plain pointer arrays, so everything except the CUDA-IPC mapping is exercised on ONE GPU: the "peers" of the
loop-back tests are separate buffers of the same device. The two-process test needs 2 GPUs; bench.py repeats
its check (`dp_parity`) at every N > 1."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from _mp import spawn_ranks

pytestmark = pytest.mark.gpu

DIN, D = 192, 512


def _arr(tensors):
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


@pytest.mark.parametrize("stream_k", [False, True])
@pytest.mark.parametrize("world", [1, 2, 8])
@pytest.mark.parametrize("shape", [(512, 192, 300), (512, 512, 1000), (4096, 4096, 2048)])
def test_scatter_gemm_matches_local_gemm_bit_exactly(world, shape, stream_k):
    from thinkdiff_mlre_b200 import _lib as L
    from thinkdiff_mlre_b200 import ops

    M, N, K = shape
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn((K, M), generator=g, device="cuda").to(torch.bfloat16)  # MN-major operands: [K, rows]
    B = torch.randn((K, N), generator=g, device="cuda").to(torch.bfloat16)
    want = ops.gemm_f32out(A, B, True, True, alpha=0.5, cta_pair=True, stream_k=stream_k)
    parts = [torch.full((M // world, N), float("nan"), device="cuda") for _ in range(world)]
    ws, ws_bytes = ops.gemm_workspace(A.device, stream_k)
    L.check(L.lib().td_gemm_tn_scatter(L.ptr(A), M, L.ptr(B), N, M, N, K, 0.5, _arr(parts), world, -1, L.ptr(ws), ws_bytes, L.stream_ptr()),
            "td_gemm_tn_scatter")
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(parts), want)  # same schedule, same accumulation order: same bits as the local-output GEMM
    # the data-parallel step's tile order (grouped by owner, rotated by rank): every output element is still stored exactly once;
    # which tiles the stream-K tail cuts along K changes, so bits may differ in the last place -- never more
    for rank in sorted({0, world // 2, world - 1}):
        parts = [torch.full((M // world, N), float("nan"), device="cuda") for _ in range(world)]
        L.check(L.lib().td_gemm_tn_scatter(L.ptr(A), M, L.ptr(B), N, M, N, K, 0.5, _arr(parts), world, rank, L.ptr(ws), ws_bytes,
                                           L.stream_ptr()), "td_gemm_tn_scatter")
        torch.cuda.synchronize()
        got = torch.cat(parts)
        assert torch.isfinite(got).all()
        torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-5 * float(want.abs().max()))
        if not stream_k:
            assert torch.equal(got, want)  # whole tiles only: the order of the tiles does not change any bit


def test_flags_post_sum_and_adamw_slots_loopback():
    from thinkdiff_mlre_b200 import _lib as L

    world, n = 4, 4096
    flags = [torch.zeros(64, dtype=torch.int32, device="cuda") for _ in range(world)]
    # signal: +1 on counter `slot` of every flag array (one call per "rank" and step); wait: the local counter has reached
    # steps * world, i.e. every rank has signalled every step
    steps = 3
    for _ in range(steps):
        for _src in range(world):
            L.check(L.lib().td_peer_signal(_arr(flags), world, 32, L.stream_ptr()), "td_peer_signal")
    L.check(L.lib().td_peer_wait(C.c_void_p(flags[2].data_ptr() + 4 * 32), 1, steps * world, 5.0, L.stream_ptr()), "td_peer_wait")
    torch.cuda.synchronize()
    for f in flags:
        assert int(f[32]) == steps * world and int(f.sum()) == steps * world
    # post + sum (fixed order)
    g = torch.Generator(device="cuda").manual_seed(1)
    srcs = [torch.randn(n, generator=g, device="cuda") for _ in range(world)]
    slots = torch.zeros((world, n), device="cuda")
    for s, src in enumerate(srcs):
        L.check(L.lib().td_peer_post(L.ptr(src), _arr([slots[s]]), 1, n, L.stream_ptr()), "td_peer_post")
    out = torch.empty(n, device="cuda")
    L.check(L.lib().td_sum_slots(L.ptr(slots), n, world, L.ptr(out), n, L.stream_ptr()), "td_sum_slots")
    want = srcs[0].clone()
    for s in srcs[1:]:
        want += s
    assert torch.equal(out, want)
    # AdamW over slots == td_adamw_step on the pre-summed gradient; bf16 rows land in every destination
    p0 = torch.randn(n, generator=g, device="cuda")
    pa, pb = p0.clone(), p0.clone()
    ma, va, mb, vb = (torch.zeros(n, device="cuda") for _ in range(4))
    dst = [torch.zeros(n, dtype=torch.bfloat16, device="cuda") for _ in range(3)]
    ref_bf16 = torch.zeros(n, dtype=torch.bfloat16, device="cuda")
    for step in (1, 2):
        L.check(L.lib().td_adamw_slots_step(L.ptr(pa), L.ptr(slots), n, world, L.ptr(ma), L.ptr(va), _arr(dst), 3, n, 0.05, 1e-3, 0.9,
                                            0.999, 1e-8, step, 0.5, None, L.stream_ptr()), "td_adamw_slots_step")
        one = lambda t: (C.c_void_p * 1)(t.data_ptr())  # noqa: E731
        L.check(L.lib().td_adamw_step(1, one(pb), one(want), one(mb), one(vb), one(ref_bf16), (C.c_int64 * 1)(n), (C.c_float * 1)(0.05),
                                      1e-3, 0.9, 0.999, 1e-8, step, 0.5, None, L.stream_ptr()), "td_adamw_step")
    torch.cuda.synchronize()
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb)
    for t in dst:
        assert torch.equal(t, ref_bf16)


def test_folded_signal_and_small_post_loopback():
    """td_peer_fold: the finisher stores the small vectors into every "rank"'s slot as it writes them, and each scattered
    weight-gradient GEMM bumps its counter at every "rank" exactly once, after all of its stores (here: buffers of one device)."""
    import thinkdiff_mlre_b200 as td
    from thinkdiff_mlre_b200 import _lib as L
    from thinkdiff_mlre_b200 import ops

    world, M = 4, 300
    torch.manual_seed(0)
    m = td.ThinkDiffAligner(DIN, D).cuda()
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn((M, DIN), generator=gen, device="cuda").to(torch.bfloat16)
    tgt = torch.randn((M, D), generator=gen, device="cuda").to(torch.bfloat16)
    W1b, b1b, W2b, b2b = m._bf16_params()
    g = m[3].weight.detach()
    _, saved = ops.aligner_mse_fwd(x, W1b, b1b, W2b, b2b, g, m.eps, tgt, defer_loss=True)
    # reference: the same backward with local outputs
    ref = ops.AlignerBackwardFromDh2(x, saved, W2b, None, grad_scale=1.0 / world)
    rsmall = torch.zeros(3 * D, device="cuda")
    rdW1, rdW2 = torch.empty((D, DIN), device="cuda"), torch.empty((D, D), device="cuda")
    ref.gelu_and_small(rsmall[2 * D :], rsmall[:D], rsmall[D : 2 * D])
    ref.gelu_linear1_and_small(rdW1, rsmall[2 * D :], rsmall[:D], rsmall[D : 2 * D])
    ref.linear2_only(rdW2)
    # folded: four launches, no separate post / signal kernels
    flags = [torch.zeros(64, dtype=torch.int32, device="cuda") for _ in range(world)]
    slots = [torch.full((3 * D,), float("nan"), device="cuda") for _ in range(world)]
    p1 = [torch.full((D // world, DIN), float("nan"), device="cuda") for _ in range(world)]
    p2 = [torch.full((D // world, D), float("nan"), device="cuda") for _ in range(world)]
    small = torch.zeros(3 * D, device="cuda")
    flag_arr, slot_arr = _arr(flags), _arr(slots)
    bwd = ops.AlignerBackwardFromDh2(x, saved, W2b, None, grad_scale=1.0 / world)
    bwd.gelu_and_small_scatter(small[2 * D :], small[:D], small[D : 2 * D], world,
                               L.PeerFold(None, -1, C.cast(slot_arr, C.c_void_p), C.c_void_p(small.data_ptr()), small.numel()))
    bwd.linear1_only_scatter(_arr(p1), world, 1, L.PeerFold(C.cast(flag_arr, C.c_void_p), 0, None, None, 0))
    bwd.linear2_only_scatter(_arr(p2), world, 1, L.PeerFold(C.cast(flag_arr, C.c_void_p), 32, None, None, 0))
    bwd.linear2_only_scatter(_arr(p2), world, 2, L.PeerFold(C.cast(flag_arr, C.c_void_p), 32, None, None, 0))  # a second GEMM: +1 again
    torch.cuda.synchronize()
    for f in flags:
        assert int(f[0]) == 1 and int(f[32]) == 2 and int(f.sum()) == 3
    assert torch.equal(small, rsmall)
    for sl in slots:
        assert torch.equal(sl, small)
    torch.testing.assert_close(torch.cat(p1), rdW1, rtol=1e-5, atol=1e-5 * float(rdW1.abs().max()))
    torch.testing.assert_close(torch.cat(p2), rdW2, rtol=1e-5, atol=1e-5 * float(rdW2.abs().max()))


def _train(rank, world, init, mode, ret):
    import torch.distributed as dist

    import thinkdiff_mlre_b200 as td
    from oracle import aligner_ref

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=init, rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        m = td.ThinkDiffAligner(DIN, D).cuda()
        m.load_state_dict(aligner_ref.init_params_numpy(DIN, D, seed=3))
        m.enable_data_parallel(defer_wait=True, sharded=mode != "plain", peer=mode == "peer")
        step = td.AlignerTrainStep(m, td.FusedAdamW(m, lr=1e-3), pipelined=True)
        losses = []
        for j in range(4):
            b = td.synthetic_lvlm_batch(4, 50, DIN, D, seed=10 * j + rank, pin=False)
            losses.append(step.step_device(b.flat.cuda(), b.src_row_start.cuda(), b.lens.cuda(), b.total_rows, b.l_max,
                                           b.extras["flat_target"].cuda()))
        step.flush()
        torch.cuda.synchronize()
        ret.put((rank, [p.detach().float().cpu().numpy() for p in m.parameters()], [float(l) for l in losses]))
    finally:
        dist.destroy_process_group()


def _run(world, mode):
    res = spawn_ranks(_train, world, (mode,))
    return {r: (params, losses) for r, params, losses in res}


def test_peer_training_world1_equals_plain_pipeline():
    """Degenerate single-rank case: every kernel of the peer path runs (scatter epilogue, flags, slot AdamW), no IPC."""
    plain, peer = _run(1, "plain"), _run(1, "peer")
    for a, b in zip(plain[0][0], peer[0][0]):
        np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(plain[0][1], peer[0][1], rtol=1e-6)


def test_peer_training_two_gpus_equals_sharded_nccl_and_keeps_replicas_identical():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sharded, peer = _run(2, "sharded"), _run(2, "peer")
    for a, b in zip(peer[0][0], peer[1][0]):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(sharded[0][0], peer[0][0]):
        np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(sharded[0][1], peer[0][1], rtol=1e-6)
