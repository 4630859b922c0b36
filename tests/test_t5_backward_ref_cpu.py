"""Pins tests/_t5_backward_ref.py on the CPU, in float64 at small shapes, to the references the rest of the suite already trusts:
the attention stages to ``_t5_attention_ref.attention_packed`` under autograd, the head and its cross-entropy to
``oracle.t5_head_ref``, and the staged sublayer backward chains (FFN, self- and cross-attention) to autograd through
``_t5_ffn_ref`` / ``_t5_decoder_block_ref``. Also checks that the deliberately wrong references the GPU test uses to show its bounds
can fail really differ from the right one."""
import numpy as np
import torch

import _t5_attention_ref
import _t5_backward_ref as B
import _t5_decoder_block_ref as blk
import _t5_ffn_ref
from thinkdiff_mlre_b200.t5 import interleave_pairs

F64 = torch.float64
H = 2
INNER = 64 * H


def _rand(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed), dtype=F64) * scale


def _bf(t):
    return t.to(torch.bfloat16).to(F64)


def _autograd_attention(q, k, v, cu_q, cu_k, bias, dout):
    qs, ks, vs = (t.float().requires_grad_(True) for t in (q, k, v))
    o, lse = _t5_attention_ref.attention_packed(qs, ks, vs, cu_q, cu_k, H, bias, return_lse=True)
    o.backward(dout.float())
    return o.detach().double(), lse.detach().double(), qs.grad.double(), ks.grad.double(), vs.grad.double()


def _close(a, b, rel=1e-5):
    scale = max(float(b.abs().max()), 1e-30)
    assert float((a - b).abs().max()) <= rel * scale, float((a - b).abs().max()) / scale


def test_self_attention_stages_match_autograd_through_the_distance_clamp():
    lens = [1, 5, 9, 3]  # n_dist 4: the clamp min(i - j, 3) is reached in the samples of 5 and 9
    cu = np.cumsum([0] + lens).tolist()
    M = cu[-1]
    q, k, v, dout = (_bf(_rand((M, INNER), s, 0.5)) for s in (1, 2, 3, 4))
    bias = _rand((H, 4), 5).float()
    o, lse, dq, dk, dv = _autograd_attention(q, k, v, cu, None, bias, dout)
    r = B.attention(q, k, v, cu, None, H, bias, dout=dout)
    for name, want in (("o", o), ("lse", lse), ("dq", dq), ("dk", dk), ("dv", dv)):
        _close(r[name], want)
        assert bool((r[name + "_arith"] >= 0).all()) and bool(torch.isfinite(r[name + "_arith"]).all())
    # staged on given O / lse: the same, when they are the exact ones
    r2 = B.attention(q, k, v, cu, None, H, bias, o_k=r["o"], lse_k=r["lse"], dout=dout)
    for name in ("dq", "dk", "dv"):
        assert torch.allclose(r2[name], r[name], rtol=0, atol=1e-14)
    # the wrong references differ from the right one on the rows they affect
    for mutate, drop in (("mask", False), ("bias", False)):
        w = B.attention(q, k, v, cu, None, H, bias, dout=dout, mutate=mutate, drop_last_tile=drop)
        assert float((w["o"] - r["o"]).abs().max()) > 1e-3 and float((w["dq"] - r["dq"]).abs().max()) > 1e-3


def test_cross_attention_stages_match_autograd_with_empty_samples():
    lq, lk = [3, 0, 1, 4, 2], [5, 4, 0, 1, 7]  # a sample with keys but no queries, one with a query but no keys
    cu_q, cu_k = np.cumsum([0] + lq).tolist(), np.cumsum([0] + lk).tolist()
    q, dout = _bf(_rand((cu_q[-1], INNER), 6, 0.5)), _bf(_rand((cu_q[-1], INNER), 7))
    k, v = _bf(_rand((cu_k[-1], INNER), 8, 0.5)), _bf(_rand((cu_k[-1], INNER), 9))
    o, lse, dq, dk, dv = _autograd_attention(q, k, v, cu_q, cu_k, None, dout)
    r = B.attention(q, k, v, cu_q, cu_k, H, dout=dout)
    for name, want in (("o", o), ("dq", dq), ("dk", dk), ("dv", dv)):
        _close(r[name], want)
    fin = torch.isfinite(lse)
    assert torch.equal(fin, torch.isfinite(r["lse"])) and torch.allclose(r["lse"][fin], lse[fin], atol=1e-5)
    # exact zeros: O and dQ of the query without keys, dK / dV of the keys no query sees; their bounds are 0
    for name, rows in (("o", slice(3, 4)), ("dq", slice(3, 4)), ("dk", slice(5, 9)), ("dv", slice(5, 9))):
        assert not bool(r[name][rows].any()) and not bool(r[name + "_arith"][rows].any())
        err, tol = B.attention_error(r[name], r, name)
        assert bool((err <= tol).all())


def test_head_and_cross_entropy_match_the_oracle():
    from oracle import t5_head_ref

    R, K, V = 7, 64, 96
    seq, W = _bf(_rand((R, K), 10)), _bf(_rand((V, K), 11, 0.3))
    labels = torch.tensor([0, -100, V - 1, 5, -100, 90, 17])
    for gs in (1.0, 3.0):
        loss, dseq, logits = t5_head_ref.lm_head_ce_fwd_bwd(seq.float().numpy(), W.float().numpy(), labels.numpy(), gs)
        z = torch.from_numpy(logits).double()
        n_valid = int((labels != -100).sum())
        ce = B.ce_rows(z, labels, gs, n_valid)
        assert abs(float(ce["loss_row"].sum()) / n_valid - float(loss)) <= 1e-6 * abs(float(loss))
        dz = B.bf16(ce["dz"])
        err, tol = B.dlogits_error(dz, ce)
        assert bool((err <= tol).all())
        assert not bool(dz[labels == -100].any())
        acc, bound = B.contract(dz, W)
        # the oracle rounds its fp32 dlogits to bf16 and contracts in fp32: within one ulp of the float64 staged value
        ref = torch.from_numpy(dseq).double()
        assert bool(((B.bf16(acc) - ref).abs() <= B.ulp(ref.abs()) + bound).all())
        # the wrong references are rejected: the label shifted by one, n_valid counting the ignored rows
        err, tol = B.dlogits_error(dz, B.ce_rows(z, torch.where(labels >= 0, (labels + 1) % V, labels), gs, n_valid))
        assert bool((err > tol).any(1)[labels != -100].all())
        err, tol = B.dlogits_error(dz, B.ce_rows(z, labels, gs, R))
        assert float((err > tol)[labels != -100].double().mean()) > 0.9


def test_ffn_backward_chain_matches_autograd():
    M, d, d_ff, eps = 5, 64, 96, 1e-6
    x, dy = _rand((M, d), 12), _rand((M, d), 13)
    ln_w, wi0, wi1, wo = 1 + 0.1 * _rand((d,), 14), _rand((d_ff, d), 15, 0.2), _rand((d_ff, d), 16, 0.2), _rand((d, d_ff), 17, 0.1)
    _, dx_want = _t5_ffn_ref.layer_ff_with_grad(x, ln_w, wi0, wi1, wo, eps, dy)
    rstd = torch.rsqrt(x.pow(2).mean(1) + eps)
    xn = ln_w * x * rstd[:, None]
    ab = interleave_pairs(xn @ wi0.T, xn @ wi1.T, dim=1)
    d_ab, tol = B.dgated(ab, dy @ wo, torch.zeros(M, d_ff, dtype=F64))
    assert bool((tol >= 0).all())
    dxn = d_ab @ interleave_pairs(wi0, wi1, dim=0)
    dx, arith = B.residual_norm_bwd(dy, x, rstd, ln_w, dxn)
    assert torch.allclose(dx, dx_want, rtol=0, atol=1e-12) and bool((arith >= 0).all())


def _block_weights(d, seed):
    names = ["layer.0.SelfAttention." + n + ".weight" for n in "qkvo"] + ["layer.1.EncDecAttention." + n + ".weight" for n in "qkvo"]
    w = {n: _rand((d, INNER) if n.endswith("o.weight") else (INNER, d), seed + i, 0.1) for i, n in enumerate(names)}
    w["layer.0.layer_norm.weight"] = 1 + 0.1 * _rand((d,), seed + 20)
    w["layer.1.layer_norm.weight"] = 1 + 0.1 * _rand((d,), seed + 21)
    return w


def test_self_attention_sublayer_backward_chain_matches_autograd():
    d, eps, lens = 128, 1e-6, [3, 6]
    cu = np.cumsum([0] + lens).tolist()
    M = cu[-1]
    w = _block_weights(d, 30)
    bias = _rand((H, 4), 31).float()
    x, dy = _rand((M, d), 32), _rand((M, d), 33)
    _, dx_want, _ = blk.with_grads(lambda xr, _: blk.self_attention_layer(xr, w, cu, H, bias, eps), x, None, dy)
    a = "layer.0.SelfAttention."
    rstd = torch.rsqrt(x.pow(2).mean(1) + eps)
    xn = w["layer.0.layer_norm.weight"] * x * rstd[:, None]
    q, k, v = (xn @ w[a + n + ".weight"].T for n in "qkv")
    d_o = dy @ w[a + "o.weight"]
    r = B.attention(q, k, v, cu, None, H, bias, dout=d_o)
    dxn = torch.cat((r["dq"], r["dk"], r["dv"]), 1) @ torch.cat([w[a + n + ".weight"] for n in "qkv"])
    dx, _ = B.residual_norm_bwd(dy, x, rstd, w["layer.0.layer_norm.weight"], dxn)
    _close(dx, dx_want)  # the block reference runs its attention core in fp32


def test_cross_attention_sublayer_backward_chain_matches_autograd():
    d, eps, lq, lk = 128, 1e-6, [2, 0, 4], [3, 2, 5]
    cu_q, cu_k = np.cumsum([0] + lq).tolist(), np.cumsum([0] + lk).tolist()
    w = _block_weights(d, 40)
    x, dy, enc = _rand((cu_q[-1], d), 41), _rand((cu_q[-1], d), 42), _rand((cu_k[-1], d), 43)
    _, dx_want, denc_want = blk.with_grads(lambda xr, er: blk.cross_attention_layer(xr, er, w, cu_q, cu_k, H, eps), x, enc, dy)
    a = "layer.1.EncDecAttention."
    rstd = torch.rsqrt(x.pow(2).mean(1) + eps)
    xn = w["layer.1.layer_norm.weight"] * x * rstd[:, None]
    q, k, v = xn @ w[a + "q.weight"].T, enc @ w[a + "k.weight"].T, enc @ w[a + "v.weight"].T
    r = B.attention(q, k, v, cu_q, cu_k, H, dout=dy @ w[a + "o.weight"])
    dx, _ = B.residual_norm_bwd(dy, x, rstd, w["layer.1.layer_norm.weight"], r["dq"] @ w[a + "q.weight"])
    d_enc, _ = B.contract(torch.cat((r["dk"], r["dv"]), 1), torch.cat((w[a + "k.weight"], w[a + "v.weight"])))
    _close(dx, dx_want)
    _close(d_enc, denc_want)
