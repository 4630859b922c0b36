"""Multi-GPU (NCCL) data-parallel parity: world-size-2 run of the real kernels with the built-in bucketed all-reduce
(overlapped and not) must equal the mean of the per-shard oracle gradients (DDP semantics). Skipped with < 2 GPUs."""
import os

import numpy as np
import pytest
import torch

from _mp import spawn_ranks

pytestmark = pytest.mark.gpu

DIN, D, SEQS = 192, 512, 6
NAMES = ("dW1", "db1", "dW2", "db2", "dg")
KEYS = ("0.weight", "0.bias", "2.weight", "2.bias", "3.weight")


def _batch():
    rng = np.random.RandomState(7)
    lens = [40, 7, 130, 64, 1, 99]
    xs = [torch.from_numpy(rng.standard_normal((n, DIN)).astype(np.float32)).to(torch.bfloat16) for n in lens]
    ts = [torch.from_numpy(rng.standard_normal((n, D)).astype(np.float32)) for n in lens]
    return xs, ts


def _worker(rank, world, init, overlap, ret):
    import torch.distributed as dist

    import thinkdiff_mlre_b200 as td
    from oracle import aligner_ref
    from thinkdiff_mlre_b200.sharding import shard_bounds

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=init, rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        m = td.ThinkDiffAligner(DIN, D).cuda()
        m.load_state_dict(aligner_ref.init_params_numpy(DIN, D, seed=3))
        m.enable_data_parallel(overlap=overlap)
        xs, ts = _batch()
        lo, hi = shard_bounds(SEQS, world, rank)
        x, t = torch.cat(xs[lo:hi]).cuda(), torch.cat(ts[lo:hi]).cuda()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = m.forward_packed(x)
        loss, dy = td.ops.masked_mse_fwd_bwd(y, t)  # this rank's OWN mean loss
        y.backward(dy)
        torch.cuda.synchronize()
        if rank == 0:
            ret.put([p.grad.float().cpu().numpy() for p in m.parameters()])
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("overlap", [True, False])
def test_two_gpu_bucketed_allreduce_equals_oracle_mean(overlap):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from oracle import aligner_ref
    from thinkdiff_mlre_b200.sharding import shard_bounds

    world = 2
    got = spawn_ranks(_worker, world, (overlap,), results=1)[0]
    params = aligner_ref.init_params_numpy(DIN, D, seed=3)
    xs, ts = _batch()
    want = None
    for r in range(world):
        lo, hi = shard_bounds(SEQS, world, r)
        x, t = torch.cat(xs[lo:hi]).float(), torch.cat(ts[lo:hi])
        fwd = aligner_ref.aligner_fwd_bwd_manual(x, params, regime="bf16")
        out = aligner_ref.aligner_fwd_bwd_manual(x, params, dy=2 * (fwd["y"] - t) / t.numel(), regime="bf16")
        g = [out[n] / world for n in NAMES]
        want = g if want is None else [a + b for a, b in zip(want, g)]
    for a, b, n in zip(got, want, NAMES):
        err = np.linalg.norm(a - b.numpy()) / np.linalg.norm(b.numpy())
        assert err < 2e-2, (n, err)


def _train_worker(rank, world, init, pipelined, sharded, ret):
    import torch.distributed as dist

    import thinkdiff_mlre_b200 as td
    from oracle import aligner_ref

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=init, rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        m = td.ThinkDiffAligner(DIN, D).cuda()
        m.load_state_dict(aligner_ref.init_params_numpy(DIN, D, seed=3))
        m.enable_data_parallel(defer_wait=True, sharded=sharded)
        step = td.AlignerTrainStep(m, td.FusedAdamW(m, lr=1e-3), pipelined=pipelined)
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


def test_two_gpu_pipelined_training_equals_sequential_and_keeps_replicas_in_sync():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = {}
    for pipelined in (False, True, "sharded"):
        res = spawn_ranks(_train_worker, 2, (bool(pipelined), pipelined == "sharded"))
        out[pipelined] = {r: (params, losses) for r, params, losses in res}
    for pipelined in (False, True, "sharded"):  # replicas stay identical (same averaged gradients on every rank)
        for a, b in zip(out[pipelined][0][0], out[pipelined][1][0]):
            np.testing.assert_array_equal(a, b)
    for mode in (True, "sharded"):  # neither pipelining nor row-sharding the optimizer changes the arithmetic
        for a, b in zip(out[False][0][0], out[mode][0][0]):
            np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(out[False][0][1], out[mode][0][1], rtol=1e-6)
