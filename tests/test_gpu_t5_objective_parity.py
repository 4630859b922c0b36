"""Per-element float64 parity of the T5 objective's backward at Flan-T5-XXL width (d 4096, H 64, d_kv 64, d_ff 10240, V 32128):
the output head and cross-entropy (``ops.lm_head_ce``), the attention core in both directions (``ops.t5_attention_fwd`` / ``_bwd``)
and the input gradients of the three decoder sublayers. Every stage is compared, element by element, with the float64 reference of
tests/_t5_backward_ref.py built from the kernels' own outputs of the stage before, within bounds derived there from the kernels'
arithmetic. The stream-K tail classes of the long GEMMs are asserted from ``td_gemm_schedule`` at run time, and for every GEMM in a
split class the same check rejects its shared tail tile rebuilt with one contributor's k-range dropped or doubled; the attention
checks reject a causal mask shifted by one, the bias read one distance off and a dropped key tile; the dlogits check rejects the
label shifted by one and an n_valid that counts ignored rows. Each test prints one JSON report line."""
import numpy as np
import pytest
import torch

import _aligner_step_ref as R
import _t5_backward_ref as B
from _parity_report import Report, shared_tile, tail_class, workers

pytestmark = pytest.mark.gpu

D, H, D_FF, V = 4096, 64, 10240, 32128
INNER = 64 * H
EPS = 1e-6
TAG = "T5_OBJECTIVE_PARITY"
# tail classes of (dseq, logits) on 74 CTA pairs
HEAD_CLASSES = {1: ("split(5)", "split(2)"), 300: ("split(3)", "split(1)"), 4340: ("split(2)", "tail unsplit"),
                4736: ("split(8)", "split(1)"), 9472: ("no tail", "no tail")}
# bench.py's first cfg2 batch: t5_labels(64, V, seed=200) packs 4340 decoder rows, synthetic_lvlm_batch(64, 256, 3584, 4096, seed=1)
# 9166 aligner rows
CFG2_MQ, CFG2_MK = 4340, 9166


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(shape, seed, scale=1.0, dtype=torch.bfloat16):
    return (torch.randn(shape, generator=_gen(seed), device="cuda") * scale).to(dtype)


def assert_class(M, N, K, want):
    got = tail_class(M, N, K, workers())
    assert got == want, f"GEMM [{M}, {K}] x [{K}, {N}]: tail class {got}, this case is meant to cover {want}"


def check_tile_can_fail(rep, name, a, w, M, N, K, epilogue):
    """The first shared tail tile of out = a w (a [M, K], w [K, N]) with its smallest contributor's k-range dropped, and added twice,
    must be rejected by the element check on at least 90 % of its elements (float64 arithmetic on reference tensors only)."""
    rows, cols, (k0, k1) = shared_tile(M, N, K)
    acc, bound = B.contract(a[rows], w[:, cols])
    part, _ = B.contract(a[rows, k0:k1], w[k0:k1, cols])

    def out(v):
        return R.bf16(v) if epilogue == "bf16" else v.float().double()

    err, tol = R.gemm_error(epilogue, out(acc), acc, bound)
    rep.require(bool((err <= tol).all()), f"{name}: the exact tile fails its own bound")
    for how, wrong in (("dropped", acc - part), ("doubled", acc + part)):
        err, tol = R.gemm_error(epilogue, out(wrong), acc, bound)
        frac = float((err > tol).double().mean())
        rep.info[f"{name}_{how}_rejected"] = round(frac, 4)
        rep.require(frac >= 0.9, f"{name}: a tile with one contributor's k-range {how} is rejected on only {frac:.3f} of its elements")


# ------------------------------------------------------------------------------------------------ A. output head + cross-entropy
@pytest.fixture(scope="module")
def w_lm():
    return _randn((V, D), 1, 0.04)


def head_inputs(Rn, W):
    """seq [R, d] and labels [R]: labels 0, V - 1 and one in the half-full last N tile (R > 1), every eighth row ignored, three peaked rows
    (seq = c W[label], so z[label] is about 24 above the rest and p_label about 1 - 1e-6); the cfg2 row count takes bench.py's labels.
    The other rows of dseq's first shared tail tile take labels inside its smallest contributor's k-range: the gradient of a row is
    dominated by -W[label], so that is where a dropped or doubled contribution shows in every row of the tile (none of them ignored)."""
    seq = _randn((Rn, D), 100 + Rn)
    if Rn == CFG2_MQ:
        import thinkdiff_mlre_b200 as td
        from thinkdiff_mlre_b200.synth import t5_labels

        labels, _, _ = td.pack_labels(t5_labels(64, V, seed=200), V)
        return seq, labels.cuda()
    labels = torch.randint(0, V, (Rn,), generator=_gen(200 + Rn), device="cuda")
    labels[7::8] = -100
    if HEAD_CLASSES[Rn][0].startswith("split"):
        rows, _, (k0, k1) = shared_tile(Rn, D, V)
        labels[rows] = torch.randint(k0, k1, (rows.stop - rows.start,), generator=_gen(300 + Rn), device="cuda")
    if Rn > 1:  # a single row is the shared tile's
        for r, lab in ((0, 0), (1, V - 1), (2, V - 100)):
            labels[r] = lab
    for r, c in ((3, 20.0), (4, 24.0), (5, 28.0)):
        if r < Rn:
            wl = W[labels[r]].double()
            seq[r] = (c / float(wl.pow(2).sum()) * wl).to(torch.bfloat16)
    return seq, labels


@pytest.mark.parametrize("Rn", [1, 300, 4340, 4736, 9472])
def test_lm_head_ce_per_element(w_lm, Rn):
    from thinkdiff_mlre_b200 import ops

    torch.cuda.reset_peak_memory_stats()
    assert_class(Rn, D, V, HEAD_CLASSES[Rn][0])
    assert_class(Rn, V, D, HEAD_CLASSES[Rn][1])
    W = w_lm
    gs = 3.0 if Rn in (300, 4736) else 1.0
    seq, labels = head_inputs(Rn, W)
    loss, dseq, logits = ops.lm_head_ce(seq, W, labels, gs, keep_logits=True)
    loss0, dseq0, _ = ops.lm_head_ce(seq, W, labels, gs)
    # the entry keeps its logits' gradient internal: rerun its loss kernel on its logits; dseq rebuilt from that gradient with the
    # entry's own dx GEMM must be bit-identical, so the gradient checked here is the one the entry contracted
    _, dlogits = ops.masked_ce_fwd_bwd(logits, labels, gs)
    rep = Report(f"lm_head_ce R={Rn} grad_scale={gs:g}", TAG)
    rep.require(torch.equal(loss, loss0) and torch.equal(dseq, dseq0), "the in-place path differs from keep_logits=True")
    dseq_re = ops.linear_bf16_dx(dlogits, W)
    rep.require(torch.equal(dseq_re, dseq), "dseq differs from linear_bf16_dx of the logits' gradient (same GEMM)")
    n_valid = int((labels != -100).sum())
    Wd = W.double()
    row_sum = row_arith = row_abs = 0.0
    n_equal = n_valid_el = 0
    shift_rows = nv_bad = nv_el = 0
    for sl in B.row_blocks(Rn):
        acc, bound = R.product(seq[sl], Wd)
        rep.check("logits", *R.gemm_error("bf16", logits[sl], acc, bound))
        del acc, bound
        lab = labels[sl]
        ce = B.ce_rows(logits[sl], lab, gs, n_valid)
        err, tol = B.dlogits_error(dlogits[sl], ce)
        rep.check("dlogits", err, tol)
        valid = lab != -100
        n_equal += int(((dlogits[sl].double() == R.bf16(ce["dz"])) & valid[:, None]).sum())
        n_valid_el += int(valid.sum()) * V
        row_sum += float(ce["loss_row"].sum())
        row_arith += float(ce["loss_arith"].sum())
        row_abs += float(ce["loss_row"].abs().sum())
        # wrong references: the label shifted by one; n_valid counting the ignored rows
        wrong = B.ce_rows(logits[sl], torch.where(valid, (lab + 1) % V, lab), gs, n_valid)
        e2, t2 = B.dlogits_error(dlogits[sl], wrong)
        shift_rows += int(((e2 > t2).any(1) & valid).sum())
        if n_valid < Rn:
            e2, t2 = B.dlogits_error(dlogits[sl], B.ce_rows(logits[sl], lab, gs, Rn))
            nv_bad += int(((e2 > t2) & valid[:, None]).sum())
            nv_el += int(valid.sum()) * V
        del ce, wrong, err, tol, e2, t2
    ref_loss = row_sum / n_valid
    rep.check("loss", torch.tensor(abs(float(loss) - ref_loss)), torch.tensor(B.loss_tolerance(row_arith, row_abs, Rn, n_valid)))
    rep.info["dlogits_bit_equal"] = round(n_equal / n_valid_el, 5)
    rep.require(n_equal >= 0.99 * n_valid_el, f"dlogits: only {n_equal / n_valid_el:.4f} of the valid rows' elements are bit-equal")
    rep.require(shift_rows == n_valid, f"dlogits: the label shifted by one is rejected on only {shift_rows} of {n_valid} rows")
    if nv_el:
        rep.info["dlogits_nvalid_wrong_rejected"] = round(nv_bad / nv_el, 4)
        rep.require(nv_bad >= 0.9 * nv_el, f"dlogits: n_valid counting ignored rows is rejected on only {nv_bad / nv_el:.3f}")
    acc, bound = B.contract(dlogits, Wd)
    rep.check("dseq", *R.gemm_error("bf16", dseq, acc, bound))
    del acc, bound
    if HEAD_CLASSES[Rn][0].startswith("split"):
        check_tile_can_fail(rep, "dseq", dlogits, W, Rn, D, V, "bf16")
    rep.finish()


# ------------------------------------------------------------------------------------------------ B. attention core
def decoder_bias(seed):
    """A [H, 128] fp32 bias by distance that favours near keys, as T5's learned decoder bias does: 0.5 N(0, 1) - distance / 32."""
    return torch.randn((H, 128), generator=_gen(seed), device="cuda") * 0.5 - torch.arange(128, device="cuda") / 32


def _affected(cu_q, cu_k, how, self_attn):
    """Rows (packed query indices) a wrong reference changes: "mask" every query but a sample's last, "bias" every query after a
    sample's first, "drop" the queries that see the dropped last key tile."""
    rows = []
    for b in range(len(cu_q) - 1):
        T = cu_q[b + 1] - cu_q[b]
        L = T if self_attn else cu_k[b + 1] - cu_k[b]
        if how == "mask":
            rows += range(cu_q[b], cu_q[b + 1] - 1)
        elif how == "bias":
            rows += range(cu_q[b] + 1, cu_q[b + 1])
        elif L > B.ATTN_TILE:
            first = (L - 1) // B.ATTN_TILE * B.ATTN_TILE if self_attn else 0
            rows += range(cu_q[b] + min(first, T), cu_q[b + 1])
    return torch.tensor(rows, dtype=torch.long, device="cuda")


def run_attention_case(label, lq, lk, self_attn, seed):
    from thinkdiff_mlre_b200 import ops

    torch.cuda.reset_peak_memory_stats()
    cu_q = np.cumsum([0] + lq).tolist()
    cu_k = cu_q if self_attn else np.cumsum([0] + lk).tolist()
    Mq, Mk = cu_q[-1], cu_k[-1]
    q, dout = _randn((Mq, INNER), seed, 0.35), _randn((Mq, INNER), seed + 1)
    k, v = _randn((Mk, INNER), seed + 2, 0.35), _randn((Mk, INNER), seed + 3)
    if self_attn:
        k, v = k[:Mq], v[:Mq]
    bias = decoder_bias(seed + 4) if self_attn else None
    cuq_d = torch.tensor(cu_q, dtype=torch.int32, device="cuda")
    cuk_d = None if self_attn else torch.tensor(cu_k, dtype=torch.int32, device="cuda")
    mq, mk = max(lq), max(lq if self_attn else lk)
    o, lse = ops.t5_attention_fwd(q, k, v, cuq_d, cuk_d, mq, mk, H, bias)
    dq, dk, dv = ops.t5_attention_bwd(dout, q, k, v, o, lse, cuq_d, cuk_d, mq, mk, H, bias)
    rep = Report(label, TAG)
    ref = B.attention(q, k, v, cu_q, None if self_attn else cu_k, H, bias, o_k=o, lse_k=lse, dout=dout)
    for name, val in (("O", o), ("lse", lse), ("dQ", dq), ("dK", dk), ("dV", dv)):
        rep.check(name, *B.attention_error(val, ref, name.lower() if name != "lse" else "lse"))
    # exact zeros: queries of samples without keys (O, dQ), keys of samples without queries (dK, dV)
    for b in range(len(cu_q) - 1):
        if cu_k[b + 1] == cu_k[b] and cu_q[b + 1] > cu_q[b]:
            rep.require(not bool(o[cu_q[b] : cu_q[b + 1]].any()) and not bool(dq[cu_q[b] : cu_q[b + 1]].any()),
                        f"sample {b} has no keys but nonzero O / dQ")
        if cu_q[b + 1] == cu_q[b] and cu_k[b + 1] > cu_k[b]:
            rep.require(not bool(dk[cu_k[b] : cu_k[b + 1]].any()) and not bool(dv[cu_k[b] : cu_k[b + 1]].any()),
                        f"sample {b}'s keys are seen by no query but have nonzero dK / dV")
    del ref
    # the bounds can fail: each wrong reference is rejected on >= 90 % of the (row, head) pairs it changes, for O and dQ
    for how in (("mask", "bias", "drop") if self_attn else ("drop",)):
        rows = _affected(cu_q, cu_k, how, self_attn)
        if rows.numel() == 0:
            continue
        wrong = B.attention(q, k, v, cu_q, None if self_attn else cu_k, H, bias, o_k=o, lse_k=lse, dout=dout,
                            mutate=how if how != "drop" else None, drop_last_tile=how == "drop")
        for name, val in (("o", o), ("dq", dq)):
            err, tol = B.attention_error(val, wrong, name)
            bad = (err > tol).reshape(Mq, H, 64).any(-1)[rows]
            frac = float(bad.double().mean())
            rep.info[f"{name}_{how}_rejected"] = round(frac, 4)
            rep.require(frac >= 0.9, f"{name}: the reference with {how} wrong is rejected on only {frac:.3f} of the rows it changes")
        del wrong
    rep.info["rows"] = [Mq, Mk]
    rep.finish()


def test_attention_core_self_per_element():
    """Causal self-attention at H 64: the production decoder lengths U{8..128}, samples of 129 and 300 (the distance clamp
    min(i - j, 127) and a third query tile), and samples of 1 and 128 rows."""
    g = torch.Generator().manual_seed(7)
    lens = torch.randint(8, 129, (40,), generator=g).tolist() + [129, 300, 1, 128]
    run_attention_case("attention self", lens, None, True, 10)


def test_attention_core_cross_per_element():
    """Cross-attention at H 64: production pairs (queries U{8..128}, keys U{1..256}) and key lengths 0, 1, 127, 128, 129, 256 and 1000
    with query lengths 1 and 128, plus a sample with keys but no queries."""
    g = torch.Generator().manual_seed(8)
    lq = torch.randint(8, 129, (24,), generator=g).tolist()
    lk = torch.randint(1, 257, (24,), generator=g).tolist()
    edge = [(5, 0), (1, 1), (128, 1), (1, 127), (128, 127), (1, 128), (128, 128), (128, 129), (1, 256), (128, 256), (1, 1000),
            (128, 1000), (0, 200), (1, 0), (128, 0)]
    lq += [a for a, _ in edge]
    lk += [b for _, b in edge]
    run_attention_case("attention cross", lq, lk, False, 20)


# ------------------------------------------------------------------------------------------------ C. sublayer input gradients
@pytest.fixture(scope="module")
def cfg2_rows():
    import thinkdiff_mlre_b200 as td
    from thinkdiff_mlre_b200.synth import t5_labels

    _, lens_q, max_q = td.pack_labels(t5_labels(64, V, seed=200), V)
    fb = td.synthetic_lvlm_batch(64, 256, 3584, 4096, seed=1, pin=False, with_target=False)
    cu_q = np.cumsum([0] + lens_q.tolist()).tolist()
    cu_k = np.cumsum([0] + fb.lens.tolist()).tolist()
    assert cu_q[-1] == CFG2_MQ and cu_k[-1] == CFG2_MK
    return cu_q, max_q, cu_k, int(fb.l_max)


def sublayer_inputs(M, seed):
    x = _randn((M, D), seed)
    dy = _randn((M, D), seed + 1, 2.0 ** -10)
    ln_w = 1 + 0.1 * torch.randn((D,), generator=_gen(seed + 2), device="cuda")
    return x, dy, ln_w


def check_dx(rep, dx, dy, x, rstd, ln_w, dxn):
    for sl in B.row_blocks(x.shape[0]):
        ref, arith = B.residual_norm_bwd(dy[sl], x[sl], rstd[sl], ln_w, dxn[sl])
        rep.check("dx", *B.bf16_out_error(dx[sl], ref, arith, ulps=1.0))


def check_d_o(rep, d_o, dy, wo):
    wt = wo.double().T
    for sl in B.row_blocks(dy.shape[0]):
        acc, bound = R.product(dy[sl], wt)
        rep.check("d_o", *R.gemm_error("bf16", d_o[sl], acc, bound))


def test_self_attention_sublayer_backward_per_element(cfg2_rows):
    from thinkdiff_mlre_b200 import ops

    torch.cuda.reset_peak_memory_stats()
    cu_q, max_q, _, _ = cfg2_rows
    M = cu_q[-1]
    assert_class(M, D, 3 * INNER, "split(2)")
    x, dy, ln_w = sublayer_inputs(M, 30)
    w_qkv, wo = _randn((3 * INNER, D), 33, 0.02), _randn((D, INNER), 34, 0.02)
    bias = decoder_bias(35)
    cuq_d = torch.tensor(cu_q, dtype=torch.int32, device="cuda")
    _, rstd, qkv, o, lse = ops.t5_self_attention_layer_fwd(x, w_qkv, wo, ln_w, EPS, bias, cuq_d, max_q, H)
    dx, dqkv = ops.t5_self_attention_layer_bwd(dy, x, rstd, qkv, o, lse, w_qkv, wo, ln_w, bias, cuq_d, max_q, H, want_dqkv=True)
    # the same backward from public calls: the d_o GEMM, the attention backward into column slices, the dxn GEMM
    d_o = ops.linear_bf16_dx(dy, wo)
    buf = torch.empty_like(dqkv)
    ops.t5_attention_bwd(d_o, qkv[:, :INNER], qkv[:, INNER : 2 * INNER], qkv[:, 2 * INNER :], o, lse, cuq_d, None, max_q, max_q, H, bias,
                         dq=buf[:, :INNER], dk=buf[:, INNER : 2 * INNER], dv=buf[:, 2 * INNER :])
    rep = Report(f"self-attention sublayer M={M}", TAG)
    rep.require(torch.equal(buf, dqkv), "dqkv from the public calls differs from the fused entry's")
    dxn = ops.linear_bf16_dx(dqkv, w_qkv)
    check_d_o(rep, d_o, dy, wo)
    ref = B.attention(qkv[:, :INNER], qkv[:, INNER : 2 * INNER], qkv[:, 2 * INNER :], cu_q, None, H, bias, o_k=o, lse_k=lse, dout=d_o)
    for i, name in enumerate(("dq", "dk", "dv")):
        rep.check("dqkv", *B.attention_error(dqkv[:, i * INNER : (i + 1) * INNER], ref, name))
    del ref
    acc, bound = B.contract(dqkv, w_qkv)
    rep.check("dxn", *R.gemm_error("bf16", dxn, acc, bound))
    del acc, bound
    check_dx(rep, dx, dy, x, rstd, ln_w, dxn)
    check_tile_can_fail(rep, "dxn", dqkv, w_qkv, M, D, 3 * INNER, "bf16")
    rep.finish()


def test_cross_attention_sublayer_backward_per_element(cfg2_rows):
    from thinkdiff_mlre_b200 import ops

    torch.cuda.reset_peak_memory_stats()
    cu_q, max_q, cu_k, max_k = cfg2_rows
    M, Mk = cu_q[-1], cu_k[-1]
    assert_class(M, D, INNER, "split(2)")
    assert_class(Mk, D, 2 * INNER, "split(2)")
    x, dy, ln_w = sublayer_inputs(M, 40)
    enc = _randn((Mk, D), 43)
    w_q, w_kv, wo = _randn((INNER, D), 44, 0.02), _randn((2 * INNER, D), 45, 0.02), _randn((D, INNER), 46, 0.02)
    cuq_d, cuk_d = (torch.tensor(c, dtype=torch.int32, device="cuda") for c in (cu_q, cu_k))
    _, rstd, q, kv, o, lse = ops.t5_cross_attention_layer_fwd(x, enc, w_q, w_kv, wo, ln_w, EPS, cuq_d, cuk_d, max_q, max_k, H)
    dx, d_enc = ops.t5_cross_attention_layer_bwd(dy, x, rstd, q, kv, o, lse, w_q, w_kv, wo, ln_w, cuq_d, cuk_d, max_q, max_k, H)
    d_o = ops.linear_bf16_dx(dy, wo)
    dkv = torch.empty((Mk, 2 * INNER), dtype=torch.bfloat16, device="cuda")
    dq, _, _ = ops.t5_attention_bwd(d_o, q, kv[:, :INNER], kv[:, INNER:], o, lse, cuq_d, cuk_d, max_q, max_k, H,
                                    dk=dkv[:, :INNER], dv=dkv[:, INNER:])
    dxn = ops.linear_bf16_dx(dq, w_q)
    # gemm_f32out with a CTA pair, K-major dkv and MN-major [Wk; Wv], stream-K on: the configuration of the entry's d_enc GEMM
    d_enc_re = ops.gemm_f32out(dkv, w_kv, False, True)
    rep = Report(f"cross-attention sublayer M={M} Mk={Mk}", TAG)
    rep.require(torch.equal(d_enc_re, d_enc), "d_enc from the public calls differs from the fused entry's")
    check_d_o(rep, d_o, dy, wo)
    ref = B.attention(q, kv[:, :INNER], kv[:, INNER:], cu_q, cu_k, H, o_k=o, lse_k=lse, dout=d_o)
    rep.check("dq", *B.attention_error(dq, ref, "dq"))
    rep.check("dkv", *B.attention_error(dkv[:, :INNER], ref, "dk"))
    rep.check("dkv", *B.attention_error(dkv[:, INNER:], ref, "dv"))
    del ref
    acc, bound = B.contract(dq, w_q)
    rep.check("dxn", *R.gemm_error("bf16", dxn, acc, bound))
    acc, bound = B.contract(dkv, w_kv)
    rep.check("d_enc", *R.gemm_error("f32", d_enc, acc, bound))
    del acc, bound
    check_dx(rep, dx, dy, x, rstd, ln_w, dxn)
    check_tile_can_fail(rep, "dxn", dq, w_q, M, D, INNER, "bf16")
    check_tile_can_fail(rep, "d_enc", dkv, w_kv, Mk, D, 2 * INNER, "f32")
    rep.finish()


def test_ffn_sublayer_backward_per_element(cfg2_rows):
    from thinkdiff_mlre_b200 import ops
    from thinkdiff_mlre_b200.t5 import interleave_pairs

    torch.cuda.reset_peak_memory_stats()
    M = cfg2_rows[0][-1]
    assert_class(M, D, 2 * D_FF, "split(2)")
    x, dy, ln_w = sublayer_inputs(M, 50)
    wi = interleave_pairs(_randn((D_FF, D), 53, 0.02), _randn((D_FF, D), 54, 0.02))
    wo = _randn((D, D_FF), 55, 0.02)
    _, rstd, ab, _ = ops.t5_ffn_fwd(x, wi, wo, ln_w, EPS)
    dx, d_ab = ops.t5_ffn_bwd(dy, x, rstd, ab, wi, wo, ln_w, want_d_ab=True)
    dxn = ops.linear_bf16_dx(d_ab, wi)
    rep = Report(f"FFN sublayer M={M}", TAG)
    wt = wo.double().T
    for sl in B.row_blocks(M):
        t, t_bound = R.product(dy[sl], wt)
        ref, arith = B.dgated(ab[sl], t, t_bound)
        rep.check("d_ab", *B.bf16_out_error(d_ab[sl], ref, arith))
        del t, t_bound, ref, arith
    acc, bound = B.contract(d_ab, wi)
    rep.check("dxn", *R.gemm_error("bf16", dxn, acc, bound))
    del acc, bound
    check_dx(rep, dx, dy, x, rstd, ln_w, dxn)
    check_tile_can_fail(rep, "dxn", d_ab, wi, M, D, 2 * D_FF, "bf16")
    rep.finish()
