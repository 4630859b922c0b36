"""Per-element float64 parity of the fused aligner train step at production width (Din 3584, D 4096), stage by stage, across the
stream-K tail classes of its five GEMMs.

The step (``AlignerTrainStep`` -> ``ThinkDiffAligner.mse_loss_backward_packed``) is run as its staged calls -- ``ops.aligner_mse_fwd``
and ``ops.AlignerBackwardFromDh2`` -- and every output is compared, element by element, with the float64 reference of
tests/_aligner_step_ref.py built from the kernels' own outputs of the stage before (so each bound is tight):

  * h0, h2 (bias-GELU / bias-sum-of-squares GEMMs): half a bf16 ulp plus the accumulation bound 2^-18 (|A| |B|^T)_ij.
    h2, rstd and the fp32 y come from ``ops.aligner_fwd``, which runs the same GEMMs (its h0 / h1 are checked bit-identical to
    the fused path's).
  * h1 against bf16(gelu(h0)) in float64: within one ulp, and at least 99.9 % bit-equal.
  * rstd, y: 1e-6 relative. dh2: one ulp plus the size of the fp32 arithmetic that forms it (which only matters where its two
    terms cancel). Loss: 1e-5 relative.
  * dh0 (DGELU GEMM; read from the backward's workspace, where the dW1 GEMM reads it): one ulp at each of its two rounding points
    plus the accumulation bound through gelu'. dW1 / db1 from the kernels' dh0, dW2 / db2 from the kernels' dh2 and h1:
    the accumulation bound, per element (dg: its column's sum of |dy xhat| and the row statistics' error). dW1 and dW2 contract
    over up to 65 k tokens, so their bound also carries an fp32 ulp of the running partial sum per MMA accumulation
    (``_aligner_step_ref.contract_rows``).
  * The bounds can fail: for every GEMM with a shared (split) tail tile, that tile rebuilt with one contributor's k-range left out,
    and with it added twice, is rejected by the same element check on at least 90 % of its elements.

The token counts are chosen for the tail class each GEMM hits on a full B200 (74 CTA pairs); the classes are asserted from the
library's host-side planner ``td_gemm_schedule`` at run time, so a planner change fails here instead of quietly moving coverage.
The whole step is checked bit-identical to the staged calls (and exactly 65536 times them with ``loss_scale=65536``), the
PDL-chained step bit-identical to a serialized one (per-launch profiling puts an event between every two kernels), and TMA
reduce-add gradient accumulation equal to the float64 sum of two micro-batches, per element.
"""
import pytest
import torch

import _aligner_step_ref as R
from _parity_report import Report, shared_tile, tail_class, workers

pytestmark = pytest.mark.gpu

DIN, D = 3584, 4096
EPS = 1e-6
GEMMS = ("fwd1", "fwd2", "dh0", "dW1", "dW2")
EPILOGUE = {"fwd1": "bf16", "fwd2": "bf16", "dh0": "dgelu", "dW1": "f32", "dW2": "f32"}
# tail class of (fwd1, fwd2, dh0, dW1, dW2) on 74 CTA pairs; "split(c)": a shared tail tile has up to c contributors
CLASSES = {
    1: ("split(1)", "split(3)", "split(3)", "tail unsplit", "tail unsplit"),
    4736: ("split(1)", "split(3)", "split(3)", "split(1)", "split(1)"),
    8224: ("split(1)", "split(3)", "split(3)", "split(2)", "split(2)"),
    8288: ("split(1)", "split(3)", "split(3)", "split(4)", "split(1)"),
    9472: ("no tail", "no tail", "no tail", "split(3)", "split(1)"),
    18944: ("no tail", "no tail", "no tail", "split(7)", "split(1)"),
    65600: ("split(2)", "split(2)", "split(2)", "split(12)", "split(3)"),
}
CFG5_M = 65600
# bench.py's first config-2 batch: synthetic_lvlm_batch(64, 256, 3584, 4096, seed=1234) packs 9130 tokens
CFG2_SEED, CFG2_M = 1234, 9130
CFG2_CLASSES = ("tail unsplit", "tail unsplit", "tail unsplit", "split(4)", "split(2)")


def gemm_mnk(name, M):
    return {"fwd1": (M, D, DIN), "fwd2": (M, D, D), "dh0": (M, D, D), "dW1": (D, DIN, M), "dW2": (D, D, M)}[name]


def assert_classes(M, want):
    got = tuple(tail_class(*gemm_mnk(g, M), workers()) for g in GEMMS)
    assert got == want, f"M={M}: tail classes {dict(zip(GEMMS, got))}, this case is meant to cover {dict(zip(GEMMS, want))}"


@pytest.fixture(scope="module")
def model():
    import thinkdiff_mlre_b200 as td
    from oracle import aligner_ref
    from thinkdiff_mlre_b200 import ops

    m = td.ThinkDiffAligner(DIN, D).cuda()
    m.load_state_dict(aligner_ref.init_params_numpy(DIN, D, seed=11))
    bf = tuple(ops.cast_to_bf16(p.detach().contiguous()) for p in (m[0].weight, m[0].bias, m[2].weight, m[2].bias))
    return m, (*bf, m[3].weight.detach())


def random_rows(M, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((M, DIN), generator=gen, device="cuda").to(torch.bfloat16)
    t = torch.randn((M, D), generator=gen, device="cuda").to(torch.bfloat16)
    return x, t


def run_staged(params, x, target, index=None, upstream=None):
    """The step's calls (mse_loss_backward_packed without data parallel): fused forward with the loss deferred, then the backward
    phases in the step's order. Returns the kernels' outputs, dh0 included."""
    from thinkdiff_mlre_b200 import ops
    from thinkdiff_mlre_b200.aligner import GradBuckets

    W1b, b1b, W2b, b2b, g = params
    loss, saved = ops.aligner_mse_fwd(x, W1b, b1b, W2b, b2b, g, EPS, target, None, index, defer_loss=True)
    bwd = ops.AlignerBackwardFromDh2(x, saved, W2b, upstream, loss_out=loss)
    gb = GradBuckets(DIN, D, x.device)
    bwd.norm_and_linear2(gb.dW2, gb.db2, gb.dg)
    bwd.gelu_and_linear1(gb.dW1, gb.db1)
    M = x.shape[0]
    off = -(-M * D * 2 // 256) * 256  # the backward workspace starts with dh2 [M, D] bf16 and dh0 [M, D] bf16, 256-byte aligned
    dh0 = bwd.ws[off : off + M * D * 2].view(torch.bfloat16).view(M, D)
    h0, h1, dh2, _ = saved
    grads = {"dW1": gb.dW1, "db1": gb.db1, "dW2": gb.dW2, "db2": gb.db2, "dg": gb.dg}
    return {"loss": loss, "h0": h0, "h1": h1, "dh2": dh2, "dh0": dh0, "grads": grads}


def forward_outputs(params, x):
    from thinkdiff_mlre_b200 import ops

    W1b, b1b, W2b, b2b, g = params
    y, (h0, h1, h2, rstd) = ops.aligner_fwd(x, W1b, b1b, W2b, b2b, g, EPS, False, True)
    return {"h0": h0, "h1": h1, "h2": h2, "rstd": rstd, "y": y}


def check_stages(params, x, t_rows, k, fwd, rep):
    """Every stage, element by element, against the float64 reference built from the previous stage's kernel output."""
    W1b, b1b, W2b, b2b, g = params
    M = x.shape[0]
    rep.require(torch.equal(fwd["h0"], k["h0"]) and torch.equal(fwd["h1"], k["h1"]),
                "aligner_fwd and aligner_mse_fwd disagree on h0 / h1 (same GEMM, same inputs)")
    W1d, W2d, b1d, b2d = (w.double() for w in (W1b, W2b, b1b, b2b))
    dy_coef = 2.0 / (M * D)
    col = {n: torch.zeros(D, dtype=torch.float64, device=x.device) for n in ("dg", "dg_tol", "db2", "db2_tol", "db1", "db1_tol")}
    loss_sum = 0.0
    n_h1_equal = n_dh2_1ulp = n_dh0_equal = 0
    for r0 in range(0, M, R.BLOCK_ROWS):
        sl = slice(r0, r0 + R.BLOCK_ROWS)
        acc, bound = R.product(x[sl], W1d, b1d)
        rep.check("fwd1", *R.gemm_error("bf16", k["h0"][sl], acc, bound))
        h0 = k["h0"][sl].double()
        ref = R.bf16(R.gelu64(h0))
        h1 = k["h1"][sl].double()
        rep.check("gelu", (h1 - ref).abs(), R.ulp(ref))
        n_h1_equal += int((h1 == ref).sum())
        acc, bound = R.product(k["h1"][sl], W2d, b2d)
        rep.check("fwd2", *R.gemm_error("bf16", fwd["h2"][sl], acc, bound))
        del acc, bound, h1, ref

        n = R.norm_mse(fwd["h2"][sl], g, t_rows[sl], EPS, dy_coef)
        rep.check("rstd", (fwd["rstd"][sl].double() - n["rstd"]).abs(), 1e-6 * n["rstd"])
        rep.check("y", (fwd["y"][sl].double() - n["y"]).abs(), 1e-6 * n["y"].abs())
        dh2 = k["dh2"][sl].double()
        err = (dh2 - n["dh2"]).abs()
        rep.check("dh2", err, R.ulp(torch.maximum(dh2.abs(), n["dh2"].abs())) + R.ROW_EPS * n["dh2_arith"])
        n_dh2_1ulp += int((err <= R.ulp(n["dh2"])).sum())
        loss_sum += float(n["diff"].pow(2).sum())
        dyx = n["dy"] * n["xhat"]
        col["dg"] += dyx.sum(0)
        col["dg_tol"] += R.ACC * dyx.abs().sum(0) + R.ROW_EPS * dy_coef * (n["y"].abs() * n["xhat"].abs()).sum(0)
        col["db2"] += dh2.sum(0)
        col["db2_tol"] += R.ACC * dh2.abs().sum(0)
        del n, dyx, err

        acc, bound = R.product(k["dh2"][sl], W2d.T)  # dh1 = dh2 W2
        err, tol = R.gemm_error("dgelu", k["dh0"][sl], acc, bound, R.gelu_grad64(h0))
        rep.check("dh0", err, tol)
        n_dh0_equal += int((err == 0).sum())
        dh0 = k["dh0"][sl].double()
        col["db1"] += dh0.sum(0)
        col["db1_tol"] += R.ACC * dh0.abs().sum(0)
        del acc, bound, err, tol, dh0, h0, dh2

    grads = k["grads"]
    acc, bound = R.contract_rows(k["dh2"], k["h1"])
    rep.check("dW2", *R.gemm_error("f32", grads["dW2"], acc, bound))
    acc, bound = R.contract_rows(k["dh0"], x)
    rep.check("dW1", *R.gemm_error("f32", grads["dW1"], acc, bound))
    del acc, bound
    for name in ("dg", "db2", "db1"):
        rep.check(name, (grads[name].double() - col[name]).abs(), col[name + "_tol"])
    ref_loss = loss_sum / (M * D)
    rep.check("loss", torch.tensor(abs(float(k["loss"]) - ref_loss)), torch.tensor(1e-5 * ref_loss))
    rep.info["h1_bit_equal"] = n_h1_equal / (M * D)
    rep.info["dh2_within_1ulp"] = n_dh2_1ulp / (M * D)
    rep.info["dh0_bit_equal"] = n_dh0_equal / (M * D)
    rep.require(n_h1_equal >= 0.999 * M * D, f"h1: only {n_h1_equal / (M * D):.5f} of the elements equal bf16(gelu(h0))")


def tile_operands(name, params, x, k, rows, cols):
    """Operands of one output tile of GEMM ``name``: A [r, K], B [c, K] (token-major A [M, r], B [M, c] for the weight gradients,
    which contract over tokens), the bias and dh0's gelu'(h0)."""
    W1b, b1b, W2b, b2b, _ = params
    if name == "fwd1":
        return x[rows], W1b[cols], b1b[cols], None
    if name == "fwd2":
        return k["h1"][rows], W2b[cols], b2b[cols], None
    if name == "dh0":
        return k["dh2"][rows], W2b[:, cols].T, None, R.gelu_grad64(k["h0"][rows, cols].double())
    if name == "dW1":
        return k["dh0"][:, rows], x[:, cols], None, None
    return k["dh2"][:, rows], k["h1"][:, cols], None, None


def check_bounds_can_fail(M, params, x, k, classes, rep):
    """For each GEMM with a shared tail tile: the tile with its smallest contributor's k-range dropped, and added twice, must be
    rejected by the element check on at least 90 % of its elements (float64 torch arithmetic only)."""
    for name, cls in zip(GEMMS, classes):
        if not cls.startswith("split"):
            continue
        rows, cols, (k0, k1) = shared_tile(*gemm_mnk(name, M))
        a, b, bias, gp = tile_operands(name, params, x, k, rows, cols)
        ep = EPILOGUE[name]
        if ep == "f32":
            acc, bound = R.contract_rows(a, b)
            part, _ = R.contract_rows(a[k0:k1], b[k0:k1])
        else:
            acc, bound = R.product(a, b, bias)
            part, _ = R.product(a[:, k0:k1], b[:, k0:k1])

        def out(v):
            return R.bf16(v) if ep == "bf16" else R.bf16(R.bf16(v) * gp) if ep == "dgelu" else v.float().double()

        err, tol = R.gemm_error(ep, out(acc), acc, bound, gp)
        rep.require(bool((err <= tol).all()), f"{name}: the exact tile fails its own bound")
        for how, wrong in (("dropped", acc - part), ("doubled", acc + part)):
            err, tol = R.gemm_error(ep, out(wrong), acc, bound, gp)
            frac = float((err > tol).double().mean())
            rep.info[f"{name}_{how}_rejected"] = round(frac, 4)
            rep.require(frac >= 0.9, f"{name}: a tile with one contributor's k-range {how} is rejected on only {frac:.3f} of its elements")


def step_device_inputs(x, t):
    """One sequence of M tokens as the step's device inputs (flat source, row starts, lengths, total rows, max length, targets)."""
    M = x.shape[0]
    return (x, torch.zeros(1, dtype=torch.int64, device="cuda"), torch.full((1,), M, dtype=torch.int32, device="cuda"), M, M, t)


def run_step(m, inputs, loss_scale=1.0):
    import thinkdiff_mlre_b200 as td

    m.zero_grad(set_to_none=True)
    loss = td.AlignerTrainStep(m, optimizer=None, loss_scale=loss_scale).step_device(*inputs)
    torch.cuda.synchronize()
    return loss.clone(), {n: p.grad.clone() for n, p in zip(("dW1", "db1", "dW2", "db2", "dg"), m.parameters())}


def run_step_serialized(m, inputs):
    """The same step with per-launch profiling on: an event recorded between every two kernels ends programmatic dependent
    launch there, so every kernel starts after its predecessor has completed."""
    from thinkdiff_mlre_b200 import _lib as L

    L.profile_enable(True)
    try:
        return run_step(m, inputs)
    finally:
        torch.cuda.synchronize()
        L.profile_enable(False)  # destroys the recorded events


def assert_bit_identical(loss, grads, k, what, factor=1.0):
    assert torch.equal(loss, k["loss"]), f"{what}: loss {float(loss)!r} != {float(k['loss'])!r}"
    for n, gr in grads.items():
        want = k["grads"][n] * factor
        assert torch.equal(gr, want), f"{what}: {n} differs on {int((gr != want).sum())} elements"


@pytest.mark.parametrize("M", [1, 4736, 8224, 8288, 9472, 18944])
def test_stage_parity_per_element_across_tail_classes(model, M):
    torch.cuda.reset_peak_memory_stats()
    assert_classes(M, CLASSES[M])
    m, params = model
    x, t = random_rows(M, seed=M)
    k = run_staged(params, x, t)
    fwd = forward_outputs(params, x)
    rep = Report(f"M={M}")
    check_stages(params, x, t, k, fwd, rep)
    check_bounds_can_fail(M, params, x, k, CLASSES[M], rep)
    rep.finish()


def test_cfg5_like_stage_parity_and_chained_step_equals_serialized(model):
    torch.cuda.reset_peak_memory_stats()
    M = CFG5_M
    assert_classes(M, CLASSES[M])
    m, params = model
    x, t = random_rows(M, seed=5)
    k = run_staged(params, x, t)
    fwd = forward_outputs(params, x)
    rep = Report(f"M={M}")
    check_stages(params, x, t, k, fwd, rep)
    check_bounds_can_fail(M, params, x, k, CLASSES[M], rep)
    del fwd
    rep.finish()
    inputs = step_device_inputs(x, t)
    loss, grads = run_step(m, inputs)
    assert_bit_identical(loss, grads, k, "step vs staged calls")
    loss, grads = run_step_serialized(m, inputs)
    assert_bit_identical(loss, grads, k, "serialized step vs staged calls")


def test_cfg2_batch_stage_parity_whole_step_loss_scale_and_serialized(model):
    import thinkdiff_mlre_b200 as td
    from thinkdiff_mlre_b200 import ops

    torch.cuda.reset_peak_memory_stats()
    m, params = model
    b = td.synthetic_lvlm_batch(64, 256, DIN, D, CFG2_SEED, pin=False)
    inputs = (b.flat.cuda(), b.src_row_start.cuda(), b.lens.cuda(), b.total_rows, b.l_max, b.extras["flat_target"].cuda())
    flat, start, lens, total, _, tgt = inputs
    x, index = ops.pack_varlen(flat, start, ops.cu_seqlens(lens), total, want_index=True)
    M = x.shape[0]
    assert M == CFG2_M
    assert_classes(M, CFG2_CLASSES)
    k = run_staged(params, x, tgt, index)
    rep = Report(f"cfg2 batch M={M}")
    check_stages(params, x, tgt[index], k, forward_outputs(params, x), rep)
    check_bounds_can_fail(M, params, x, k, CFG2_CLASSES, rep)
    rep.finish()

    loss, grads = run_step(m, inputs)
    assert_bit_identical(loss, grads, k, "step vs staged calls")
    loss, grads = run_step(m, inputs, loss_scale=65536.0)
    assert_bit_identical(loss, grads, k, "step with loss_scale=65536", factor=65536.0)
    loss, grads = run_step_serialized(m, inputs)
    assert_bit_identical(loss, grads, k, "serialized step vs staged calls")


def test_accumulated_micro_batches_equal_the_float64_sum(model):
    """Two micro-batches at a split-tail shape (dW1 and dW2 tails of 2 contributors) accumulated with accumulate_into: the TMA
    reduce-add (and the finisher's add) leaves exactly fp32(g1 + g2), per element."""
    from thinkdiff_mlre_b200.aligner import GradBuckets

    M = 8224
    assert_classes(M, CLASSES[M])
    m, params = model
    batches = [random_rows(M, seed=s) for s in (101, 102)]
    single = [run_staged(params, x, t)["grads"] for x, t in batches]
    gb = GradBuckets(DIN, D, "cuda")
    for f in gb.flats().values():
        f.zero_()
    for x, t in batches:
        m.mse_loss_backward_packed(x, t, accumulate_into=gb, set_grads=False)
    acc = dict(zip(("dW1", "db1", "dW2", "db2", "dg"), gb.in_parameter_order()))
    for n, got in acc.items():
        want = (single[0][n].double() + single[1][n].double()).float()
        assert torch.equal(got, want), f"{n}: {int((got != want).sum())} elements differ from fp32(g1 + g2)"
