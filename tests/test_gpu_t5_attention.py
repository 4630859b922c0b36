"""GPU parity of the T5 attention kernels (csrc/attn_sm100.cuh; SURVEY section 8 f-1) through the C ABI and the autograd boundary:
both modes against the fp32 oracle on the same bf16 inputs (O, LSE, dQ, dK, dV) at lengths that cross the 128-row tile edges;
against transformers' T5Attention under bf16 autocast on the padded batch; strided / fused buffers and determinism; a whole
cross-attention sublayer on packed aligner rows against T5LayerCrossAttention; and the rejected arguments.
Tolerances (relative Frobenius): O 5e-3, gradients 1e-2 against the fp32 oracle; 2e-2 against HF under autocast (BASELINE.json)."""
import pytest
import torch

import _t5_attention_ref as ref

pytestmark = pytest.mark.gpu
DK = 64


def _rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _cu(lens, dev="cuda"):
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    return cu, torch.tensor(cu, dtype=torch.int32, device=dev)


def _inputs(Mq, Mk, H, seed, scale=0.25):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = (torch.randn((Mq, H * DK), generator=g, device="cuda") * scale).to(torch.bfloat16)
    k = (torch.randn((Mk, H * DK), generator=g, device="cuda") * scale).to(torch.bfloat16)
    v = torch.randn((Mk, H * DK), generator=g, device="cuda").to(torch.bfloat16)
    do = torch.randn((Mq, H * DK), generator=g, device="cuda").to(torch.bfloat16)
    return q, k, v, do


def _table(H, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((32, H), generator=g) * 0.5).to(torch.bfloat16)


def _oracle(q, k, v, do, cu_q, cu_k, H, bias):
    qf, kf, vf = (t.detach().float().cpu().requires_grad_(True) for t in (q, k, v))
    o, lse = ref.attention_packed(qf, kf, vf, cu_q, cu_k, H, None if bias is None else bias.cpu(), return_lse=True)
    o.backward(do.float().cpu())
    return o.detach(), lse.detach(), qf.grad, kf.grad, vf.grad


LENS_K = [0, 1, 127, 128, 129, 256, 1000]
LENS_Q = [1, 64, 128, 129, 200]


@pytest.mark.parametrize("H", [4, 64])
@pytest.mark.parametrize("mode", ["cross", "self"])
def test_attention_matches_the_fp32_oracle(mode, H):
    from thinkdiff_mlre_b200 import ops
    from thinkdiff_mlre_b200.t5 import t5_position_bias_by_distance

    if mode == "cross":  # every key length against a cycling query length, plus a sample whose keys no query sees
        lens_k = LENS_K + [5]
        lens_q = [LENS_Q[i % len(LENS_Q)] for i in range(len(LENS_K))] + [0]
        bias = None
    else:
        lens_q = LENS_Q + [0, 3]
        lens_k = lens_q
        bias = t5_position_bias_by_distance(_table(H)).cuda()
    cu_q, cuq = _cu(lens_q)
    cu_k, cuk = _cu(lens_k)
    q, k, v, do = _inputs(cu_q[-1], cu_k[-1], H, seed=H + len(mode))
    o, lse = ops.t5_attention_fwd(q, k, v, cuq, None if bias is not None else cuk, max(lens_q), max(lens_k), H, bias)
    dq, dk, dv = ops.t5_attention_bwd(do, q, k, v, o, lse, cuq, None if bias is not None else cuk, max(lens_q), max(lens_k), H, bias)
    torch.cuda.synchronize()
    ro, rlse, rdq, rdk, rdv = _oracle(q, k, v, do, cu_q, cu_k, H, bias)
    errs = {"o": _rel(o, ro), "dq": _rel(dq, rdq), "dk": _rel(dk, rdk), "dv": _rel(dv, rdv)}
    assert errs["o"] <= 5e-3 and max(errs["dq"], errs["dk"], errs["dv"]) <= 1e-2, errs
    finite = torch.isfinite(rlse)
    assert torch.equal(torch.isfinite(lse.cpu()), finite)
    assert float((lse.cpu()[finite] - rlse[finite]).abs().max()) < 2e-3 * float(rlse[finite].abs().max() + 1)
    for b in range(len(lens_q)):
        if lens_k[b] == 0:  # no keys: O = 0, dQ = 0 exactly, lse = -inf
            assert not o[cu_q[b] : cu_q[b + 1]].any() and not dq[cu_q[b] : cu_q[b + 1]].any()
        if lens_q[b] == 0:  # keys no query sees: dK = dV = 0 exactly
            assert not dk[cu_k[b] : cu_k[b + 1]].any() and not dv[cu_k[b] : cu_k[b + 1]].any()


def _hf_autocast(qp, kp, vp, mask, table=None):
    from transformers import T5Config
    from transformers.models.t5.modeling_t5 import T5Attention

    class Const(torch.nn.Module):
        def __init__(self, t):
            super().__init__()
            self.t = t

        def forward(self, x):
            return self.t

    H = qp.shape[-1] // DK
    cfg = T5Config(vocab_size=16, d_model=H * DK, d_kv=DK, d_ff=32, num_layers=1, num_heads=H, relative_attention_num_buckets=32,
                   relative_attention_max_distance=128, dropout_rate=0.0, is_decoder=True, use_cache=False)
    att = T5Attention(cfg, has_relative_attention_bias=table is not None, layer_idx=0).cuda().eval()
    if table is not None:
        with torch.no_grad():
            att.relative_attention_bias.weight.copy_(table.float())
    att.q, att.k, att.v, att.o = Const(qp), Const(kp), Const(vp), torch.nn.Identity()
    hidden = torch.zeros(qp.shape, device="cuda")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        return att(hidden, mask=mask, key_value_states=None if table is not None else torch.zeros(kp.shape, device="cuda"))[0]


def _pad(x, cu, L):
    out = torch.zeros((len(cu) - 1, L, x.shape[1]), dtype=x.dtype, device=x.device)
    for b in range(len(cu) - 1):
        out[b, : cu[b + 1] - cu[b]] = x[cu[b] : cu[b + 1]]
    return out


def _unpad(xp, cu):
    return torch.cat([xp[b, : cu[b + 1] - cu[b]] for b in range(len(cu) - 1)])


@pytest.mark.parametrize("mode", ["cross", "self"])
def test_attention_vs_hf_t5_attention_under_autocast(mode):
    """Valid rows within 2e-2 of HF's padded batch + mask under bf16 autocast, and the kernel is closer to the fp32 oracle than HF's
    own autocast result is (HF rounds the unscaled scores to bf16 before the softmax; the kernel keeps them in fp32)."""
    import thinkdiff_mlre_b200 as td

    H = 8
    lens_q = [37, 128, 5, 100] if mode == "cross" else [37, 128, 5, 100]
    lens_k = [200, 17, 129, 64] if mode == "cross" else lens_q
    cu_q, cuq = _cu(lens_q)
    cu_k, cuk = _cu(lens_k)
    q, k, v, do = _inputs(cu_q[-1], cu_k[-1], H, seed=7)
    table = _table(H, seed=3) if mode == "self" else None
    bias = None if table is None else td.t5_position_bias_by_distance(table).cuda()
    T, L = max(lens_q), max(lens_k)
    qp, kp, vp = (_pad(x, c, n).requires_grad_(True) for x, c, n in ((q, cu_q, T), (k, cu_k, L), (v, cu_k, L)))
    if mode == "cross":
        mask = torch.zeros((len(lens_q), 1, 1, L), device="cuda")
        for b, n in enumerate(lens_k):
            mask[b, ..., n:] = torch.finfo(torch.float32).min
    else:
        mask = torch.full((T, T), torch.finfo(torch.float32).min, device="cuda").triu(1)[None, None]
    want = _hf_autocast(qp, kp, vp, mask, table)
    qa, ka, va = (x.clone().requires_grad_(True) for x in (q, k, v))
    got = td.t5_attention(qa, ka, va, cuq, None if mode == "self" else cuk, T, L, H, position_bias=bias)
    got.backward(do)
    want.backward(_pad(do, cu_q, T))
    ro, _, rdq, rdk, rdv = _oracle(q, k, v, do, cu_q, cu_k, H, bias)
    hf_o = _unpad(want.detach(), cu_q)
    assert _rel(got, hf_o) < 2e-2
    for g, hp, cu in ((qa.grad, qp.grad, cu_q), (ka.grad, kp.grad, cu_k), (va.grad, vp.grad, cu_k)):
        assert _rel(g, _unpad(hp, cu)) < 2e-2
        assert all(not hp[b, cu[b + 1] - cu[b] :].any() for b in range(len(cu) - 1))  # HF's pad rows: no gradient
    assert _rel(got, ro) <= _rel(hf_o, ro), (_rel(got, ro), _rel(hf_o, ro))


def test_strided_slices_fused_dkdv_and_determinism():
    from thinkdiff_mlre_b200 import ops
    from thinkdiff_mlre_b200.t5 import t5_position_bias_by_distance

    H = 4
    inner = H * DK
    lens = [129, 3, 77]
    cu, cut = _cu(lens)
    M = cu[-1]
    g = torch.Generator(device="cuda").manual_seed(11)
    qkv = (torch.randn((M, 3 * inner), generator=g, device="cuda") * 0.25).to(torch.bfloat16)
    do = torch.randn((M, inner), generator=g, device="cuda").to(torch.bfloat16)
    bias = t5_position_bias_by_distance(_table(H)).cuda()
    q, k, v = qkv[:, :inner], qkv[:, inner : 2 * inner], qkv[:, 2 * inner :]
    # self-attention on column slices of one fused [M, 3 inner] projection output
    o_s, lse_s = ops.t5_attention_fwd(q, k, v, cut, None, 129, 129, H, bias)
    o_c, lse_c = ops.t5_attention_fwd(q.contiguous(), k.contiguous(), v.contiguous(), cut, None, 129, 129, H, bias)
    assert torch.equal(o_s, o_c) and torch.equal(lse_s, lse_c)
    # cross-attention with dK | dV landing in one [Mk, 2 inner] buffer (the input gradient of a fused [Wk; Wv] projection)
    lens_k = [300, 1, 128]
    cu_k, cukt = _cu(lens_k)
    kv = torch.randn((cu_k[-1], 2 * inner), generator=g, device="cuda").to(torch.bfloat16) * 0.25
    kx, vx = kv[:, :inner], kv[:, inner:]
    o, lse = ops.t5_attention_fwd(q, kx, vx, cut, cukt, 129, 300, H)
    dkv = torch.empty_like(kv)
    dq1, dk1, dv1 = ops.t5_attention_bwd(do, q, kx, vx, o, lse, cut, cukt, 129, 300, H, dk=dkv[:, :inner], dv=dkv[:, inner:])
    dq2, dk2, dv2 = ops.t5_attention_bwd(do, q.contiguous(), kx.contiguous(), vx.contiguous(), o, lse, cut, cukt, 129, 300, H)
    assert torch.equal(dq1, dq2) and torch.equal(dkv[:, :inner], dk2) and torch.equal(dkv[:, inner:], dv2)
    # two identical calls give identical bits
    o2, lse2 = ops.t5_attention_fwd(q, kx, vx, cut, cukt, 129, 300, H)
    dq3, dk3, dv3 = ops.t5_attention_bwd(do, q, kx, vx, o2, lse2, cut, cukt, 129, 300, H)
    assert torch.equal(o, o2) and torch.equal(lse, lse2) and torch.equal(dq3, dq2) and torch.equal(dk3, dk2) and torch.equal(dv3, dv2)


def test_cross_attention_sublayer_on_packed_rows_vs_hf_t5_layer_cross_attention():
    """frozen_linear(Wq) -> frozen_linear([Wk; Wv]) on the packed aligner rows -> t5_attention -> frozen_linear(Wo), plus HF's own
    pre-norm and residual, against T5LayerCrossAttention on the zero-padded encoder batch + mask under bf16 autocast: the output and
    the gradient into the encoder rows (what flows back into the aligner); HF's pad rows get no gradient."""
    import thinkdiff_mlre_b200 as td
    from transformers import T5Config
    from transformers.models.t5.modeling_t5 import T5LayerCrossAttention

    H, D = 8, 512
    inner = H * DK
    cfg = T5Config(vocab_size=16, d_model=D, d_kv=DK, d_ff=64, num_layers=1, num_heads=H, dropout_rate=0.0, is_decoder=True, use_cache=False)
    torch.manual_seed(0)
    layer = T5LayerCrossAttention(cfg, layer_idx=0).cuda().eval()
    with torch.no_grad():
        for p in layer.parameters():
            p.copy_(torch.randn(p.shape) * 0.03 + (1.0 if p.dim() == 1 else 0.0))
    for p in layer.parameters():
        p.requires_grad_(False)
    lens_k, T = [30, 200, 1, 130], 40
    cu_k, cukt = _cu(lens_k)
    B = len(lens_k)
    g = torch.Generator(device="cuda").manual_seed(5)
    h = torch.randn((B, T, D), generator=g, device="cuda")
    enc = torch.randn((cu_k[-1], D), generator=g, device="cuda").to(torch.bfloat16).requires_grad_(True)
    L = max(lens_k)
    enc_pad = _pad(enc.detach(), cu_k, L).requires_grad_(True)
    mask = torch.zeros((B, 1, 1, L), device="cuda")
    for b, n in enumerate(lens_k):
        mask[b, ..., n:] = torch.finfo(torch.float32).min
    up = torch.randn((B, T, D), generator=g, device="cuda")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        want = layer(h, key_value_states=enc_pad, attention_mask=mask)[0]
    want.backward(up)
    a = layer.EncDecAttention
    w_kv = torch.cat([a.k.weight, a.v.weight]).to(torch.bfloat16)
    cu_q = torch.arange(0, (B + 1) * T, T, dtype=torch.int32, device="cuda")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        x = layer.layer_norm(h).reshape(B * T, D)
    qx = td.frozen_linear(x, a.q.weight.to(torch.bfloat16))
    kv = td.frozen_linear(enc, w_kv)
    att = td.t5_attention(qx, kv[:, :inner], kv[:, inner:], cu_q, cukt, T, L, H)
    got = h + td.frozen_linear(att, a.o.weight.to(torch.bfloat16)).view(B, T, D).float()
    got.backward(up)
    assert _rel(got, want) < 2e-2
    assert _rel(enc.grad, _unpad(enc_pad.grad, cu_k)) < 2e-2
    assert all(not enc_pad.grad[b, n:].any() for b, n in enumerate(lens_k))


def test_rejected_arguments_raise_with_the_library_message():
    from thinkdiff_mlre_b200 import _lib as L
    from thinkdiff_mlre_b200 import ops

    H = 4
    cu, cut = _cu([5, 9])
    q, k, v, do = _inputs(cu[-1], cu[-1], H, seed=1)
    with pytest.raises(RuntimeError, match="inner=256 must be 64 \\* H"):  # d_kv != 64
        ops.t5_attention_fwd(q, k, v, cut, cut, 9, 9, 8)
    lib, s = L.lib(), L.stream_ptr()
    o = torch.empty_like(q)
    inner = H * DK
    rc = lib.td_t5_attention_fwd(L.ptr(q), inner, L.ptr(k), inner, L.ptr(v), inner, L.ptr(cut), None, 2, H, inner, 9, 9, cu[-1], 1, None,
                                 0, L.ptr(o), inner, None, s)
    assert rc == -1 and "needs the relative position bias table" in L.last_error()
    rc = lib.td_t5_attention_fwd(L.ptr(q), inner + 4, L.ptr(k), inner, L.ptr(v), inner, L.ptr(cut), L.ptr(cut), 2, H, inner, 9, 9, cu[-1], 0,
                                 None, 0, L.ptr(o), inner, None, s)
    assert rc == -1 and "row pitches" in L.last_error()
    rc = lib.td_t5_attention_fwd(L.ptr(q), inner, L.ptr(k), inner, None, inner, L.ptr(cut), L.ptr(cut), 2, H, inner, 9, 9, cu[-1], 0,
                                 None, 0, L.ptr(o), inner, None, s)
    assert rc == -1 and "null pointer" in L.last_error()
    o, lse = ops.t5_attention_fwd(q, k, v, cut, cut, 9, 9, H)
    ws = torch.empty((16,), dtype=torch.uint8, device="cuda")
    dq, dk, dv = (torch.empty_like(q) for _ in range(3))
    rc = lib.td_t5_attention_bwd(L.ptr(do), inner, L.ptr(q), inner, L.ptr(k), inner, L.ptr(v), inner, L.ptr(cut), L.ptr(cut), 2, H, inner,
                                 9, 9, cu[-1], 0, None, 0, L.ptr(o), inner, L.ptr(lse), L.ptr(dq), inner, L.ptr(dk), inner, L.ptr(dv), inner,
                                 L.ptr(ws), 16, s)
    assert rc == -1 and "workspace too small" in L.last_error()
