"""How the GEMM schedule sizes its stream-K tail (plan_schedule in thinkdiff_mlre_b200/csrc/gemm_host.cuh), checked on the CPU
through `td_gemm_schedule`. The number of tail ranges minimises an estimate of the tail's time in k-blocks: the longest range plus
KFOLD k-blocks for each partial the busiest owner folds in. Cutting the tail as finely as kMinTailKBlocks allows made an owner
fold up to 16 partials one after another at the config-2 dW1 shape (38 at config 5)."""
import pytest

from test_gemm_schedule import KMIN, schedule

KFOLD = 8  # kTailFoldKBlocks (gemm_sm100.cuh)
WORKERS = 74  # CTA pairs on a 148-SM B200

SHAPES = {
    # the five GEMMs of a config-2 step: fwd1, fwd2 / dh0, dW2, dW1 (M x N x K, K = tokens for the weight gradients)
    "cfg2_fwd1": (8451, 4096, 3584), "cfg2_fwd2": (8451, 4096, 4096), "cfg2_dW2": (4096, 4096, 8451), "cfg2_dW1": (4096, 3584, 8451),
    "cfg5_fwd1": (67724, 4096, 3584), "cfg5_fwd2": (67724, 4096, 4096), "cfg5_dW2": (4096, 4096, 67724), "cfg5_dW1": (4096, 3584, 67724),
    # frozen T5 head and its input gradient
    "t5_head": (8192, 32128, 4096), "t5_head_dx": (8192, 4096, 32128),
}


def tail_of(segs, KB):
    """(k-blocks of the longest tail range, most ranges sharing one tail tile) of a schedule; (0, 0) without a tail."""
    tail = [s for s in segs if not (s["kind"] == 0 and s["kb0"] == 0 and s["kb1"] == KB)]
    if not tail:
        return 0, 0
    per_range, per_tile = {}, {}
    for s in tail:
        per_range[s["range"]] = per_range.get(s["range"], 0) + s["kb1"] - s["kb0"]
        per_tile.setdefault(s["tile"], set()).add(s["range"])
    return max(per_range.values()), max(len(r) for r in per_tile.values())


def old_plan_tail(M, N, K, workers):
    """The tail the schedule had before its size was chosen by cost: as many ranges of at least KMIN k-blocks as fit."""
    tiles, KB = -(-M // 256) * -(-N // 256), -(-K // 64)
    R = tiles % workers
    if R == 0:
        return 0, 0
    units = R * KB
    wt = min(max(units // KMIN, R), workers)
    q, r = divmod(units, wt)

    def worker_of(u):
        big = r * (q + 1)
        return u // (q + 1) if u < big else r + (u - big) // q

    return -(-units // wt), max(worker_of((t + 1) * KB - 1) - worker_of(t * KB) + 1 for t in range(R))


def est(longest, parts):
    return longest + KFOLD * max(parts - 1, 0)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_tail_estimate_is_never_worse_than_the_finest_cut(name):
    M, N, K = SHAPES[name]
    assert -(-M // 256) * -(-N // 256) >= WORKERS  # full waves plus a tail: the old plan is the finest cut
    new = tail_of(schedule(M, N, K, WORKERS), -(-K // 64))
    old = old_plan_tail(M, N, K, WORKERS)
    assert est(*new) <= est(*old)


@pytest.mark.parametrize("name", ["cfg2_dW1", "cfg5_dW1"])
def test_dw1_tail_is_no_longer_split_many_ways(name):
    M, N, K = SHAPES[name]
    longest, parts = tail_of(schedule(M, N, K, WORKERS), -(-K // 64))
    old_longest, old_parts = old_plan_tail(M, N, K, WORKERS)
    assert old_parts >= 17 and 2 * parts <= old_parts and longest >= old_longest
