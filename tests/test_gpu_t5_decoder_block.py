"""GPU parity of the T5 decoder's attention sublayers, block and stack on packed rows (td_t5_self_attention_layer_* /
td_t5_cross_attention_layer_*, t5_decoder_block, t5_decoder_stack): the projections and the residual GEMM on the kernels' own
intermediates; the sublayers' out, dx and d_enc against the float64 reference on the same bf16 inputs at d 512 / H 8 and d 4096 / H 64,
with decoder totals across the 128- and 256-row tile edges and the stream-K tails, samples of 1 and 128 rows and a cross sample without
aligner rows; each sublayer, one T5Block, a 3-block T5Stack and the stack -> lm_head -> CE loss against transformers under bf16
autocast (the kernels' error against float64 at most 1.25x HF's own); determinism, the inference path, M = 0, an fp32 enc whose
gradient is summed in fp32, and the rejected arguments."""
import pytest
import torch

import _t5_decoder_block_ref as ref
import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib, ops

pytestmark = pytest.mark.gpu
EPS = 1e-6
NEG = torch.finfo(torch.float32).min
_stacks = {}


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _ulp(t, floor=2.0 ** -10):
    e = torch.floor(torch.log2(t.double().abs().clamp_min(floor)))
    return torch.pow(2.0, e - 7)


def _cu(lens):
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    return cu, torch.tensor(cu, dtype=torch.int32, device="cuda")


def _pad(x, cu, L):
    out = x.new_zeros((len(cu) - 1, L, x.shape[1]))
    for b in range(len(cu) - 1):
        out[b, : cu[b + 1] - cu[b]] = x[cu[b] : cu[b + 1]]
    return out


def _unpad(xp, cu):
    return torch.cat([xp[b, : cu[b + 1] - cu[b]] for b in range(len(cu) - 1)])


def _config(d, H, d_ff, n_layers, vocab=32):
    import transformers

    return transformers.T5Config(vocab_size=vocab, d_model=d, d_kv=64, d_ff=d_ff, num_layers=n_layers, num_decoder_layers=n_layers,
                                 num_heads=H, relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                                 feed_forward_proj="gated-gelu", is_decoder=True, use_cache=False, layer_norm_epsilon=EPS)


def _hf_stack(d, H, d_ff, n_layers):
    """A frozen bf16 transformers decoder T5Stack on the GPU with seeded weights scaled so the residual stream stays O(1) and the
    attention scores O(1): q / k rows of norm ~0.25, v ~1, o and wo by 1/sqrt(fan-in), norm weights 1 + 0.1 N(0, 1). Cached."""
    key = (d, H, d_ff, n_layers)
    if key not in _stacks:
        from transformers.models.t5.modeling_t5 import T5Stack

        g = torch.Generator(device="cuda").manual_seed(d + H + d_ff + n_layers)
        with torch.device("cuda"):
            stack = T5Stack(_config(d, H, d_ff, n_layers)).eval()
        with torch.no_grad():
            for name, p in stack.named_parameters():
                r = torch.randn(p.shape, generator=g, device="cuda")
                if p.dim() == 1:
                    p.copy_(1.0 + 0.1 * r)
                elif "relative_attention_bias" in name:
                    p.copy_(0.5 * r)
                else:
                    scale = 0.25 if name.endswith(("q.weight", "k.weight")) else 1.0
                    p.copy_(r * scale * p.shape[1] ** -0.5)
        _stacks[key] = stack.to(torch.bfloat16).requires_grad_(False)
    return _stacks[key]


def _weights(stack):
    w = td.T5DecoderWeights.from_module(stack).to("cuda")
    return w, [ref.to(b.state_dict(), torch.float64) for b in stack.block], stack.final_layer_norm.weight.double()


def _bias64(w):
    return w.position_bias.double()


def _rows(lens, d, seed, dtype=torch.bfloat16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((sum(lens), d), generator=g, device="cuda").to(torch.bfloat16).to(dtype)


CASES = [  # (d, H, decoder lengths, aligner lengths)
    (512, 8, [1], [3]),
    (512, 8, [128], [1]),
    (512, 8, [1, 128], [0, 200]),
    (512, 8, [127, 128, 1], [64, 0, 5]),
    (512, 8, [100, 57, 100], [1, 128, 300]),
    (512, 8, "cfg", "cfg"),
    (4096, 64, [1, 128], [0, 200]),
    (4096, 64, [127, 128, 1], [64, 0, 5]),
    (4096, 64, "cfg", "cfg"),
]


def _lens(spec_q, spec_k, seed):
    if spec_q != "cfg":
        return spec_q, spec_k
    gen = torch.Generator().manual_seed(seed)  # 40 samples: decoder U{1..128} (~2600 rows), aligner U{0..256}
    return torch.randint(1, 129, (40,), generator=gen).tolist(), torch.randint(0, 257, (40,), generator=gen).tolist()


@pytest.mark.parametrize("case", range(len(CASES)), ids=lambda i: f"d{CASES[i][0]}_{i}")
def test_sublayers_stages_and_float64_parity(case):
    d, H, lq, lk = CASES[case]
    lens_q, lens_k = _lens(lq, lk, seed=case)
    stack = _hf_stack(d, H, 1024, 1)
    w, blocks64, _ = _weights(stack)
    bw, w64 = w.blocks[0], blocks64[0]
    cu_q, cuq = _cu(lens_q)
    cu_k, cuk = _cu(lens_k)
    M, Mk, T, L = cu_q[-1], cu_k[-1], max(lens_q), max(lens_k)
    x, enc = _rows(lens_q, d, 3 * case), _rows(lens_k, d, 3 * case + 1)
    dy = _rows(lens_q, d, 3 * case + 2)
    bias = w.position_bias

    # self-attention sublayer
    out, rstd, qkv, o, lse = ops.t5_self_attention_layer_fwd(x, bw.w_qkv, bw.wo_self, bw.ln_self, EPS, bias, cuq, T, H)
    dx, dqkv = ops.t5_self_attention_layer_bwd(dy, x, rstd, qkv, o, lse, bw.w_qkv, bw.wo_self, bw.ln_self, bias, cuq, T, H, want_dqkv=True)
    xn, rstd_n = ops.rmsnorm_fwd(x, bw.ln_self, EPS, out_bf16=True)
    assert torch.equal(rstd, rstd_n)
    want = xn.double() @ bw.w_qkv.double().t()
    assert _rel(qkv, want) <= 2e-3 and bool(((qkv.double() - want).abs() <= 2 * _ulp(want)).all())
    proj = o.double() @ bw.wo_self.double().t()
    want = (x.double() + proj.to(torch.bfloat16).double()).to(torch.bfloat16).double()
    assert bool(((out.double() - want).abs() <= _ulp(want, 2.0 ** -14) + 2 * _ulp(proj)).all())
    r_out, r_dx, _ = ref.with_grads(lambda xr, er: ref.self_attention_layer(xr, w64, cu_q, H, _bias64(w), EPS), x, None, dy)
    assert _rel(out, r_out) <= 5e-3 and _rel(dx, r_dx) <= 1e-2, (_rel(out, r_out), _rel(dx, r_dx))
    assert dqkv.shape == (M, 3 * 64 * H) and dqkv.abs().sum() > 0

    # cross-attention sublayer
    out, rstd, q, kv, o, lse = ops.t5_cross_attention_layer_fwd(x, enc, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, EPS, cuq, cuk, T, L, H)
    dx, d_enc = ops.t5_cross_attention_layer_bwd(dy, x, rstd, q, kv, o, lse, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, cuq, cuk, T, L, H)
    xn, _ = ops.rmsnorm_fwd(x, bw.ln_cross, EPS, out_bf16=True)
    for got, a, wt in ((q, xn, bw.w_q), (kv, enc, bw.w_kv)):
        want = a.double() @ wt.double().t()
        assert _rel(got, want) <= 2e-3 and bool(((got.double() - want).abs() <= 2 * _ulp(want)).all())
    proj = o.double() @ bw.wo_cross.double().t()
    want = (x.double() + proj.to(torch.bfloat16).double()).to(torch.bfloat16).double()
    assert bool(((out.double() - want).abs() <= _ulp(want, 2.0 ** -14) + 2 * _ulp(proj)).all())
    r_out, r_dx, r_denc = ref.with_grads(lambda xr, er: ref.cross_attention_layer(xr, er, w64, cu_q, cu_k, H, EPS), x, enc, dy)
    assert d_enc.dtype == torch.float32 and d_enc.shape == enc.shape
    errs = (_rel(out, r_out), _rel(dx, r_dx), _rel(d_enc, r_denc))
    assert errs[0] <= 5e-3 and errs[1] <= 1e-2 and errs[2] <= 1e-2, errs
    for b, n in enumerate(lens_k):
        if n == 0:  # no aligner rows: o = 0, out = x exactly
            assert torch.equal(out[cu_q[b] : cu_q[b + 1]], x[cu_q[b] : cu_q[b + 1]])


LQ, LK = [37, 128, 5, 100, 1], [200, 17, 129, 64, 3]


def _hf_masks(lens_q, lens_k):
    T, L = max(lens_q), max(lens_k)
    causal = torch.full((T, T), NEG, device="cuda").triu(1)[None, None].expand(len(lens_q), 1, T, T)
    enc_mask = torch.zeros((len(lens_k), 1, 1, L), device="cuda")
    for b, n in enumerate(lens_k):
        enc_mask[b, ..., n:] = NEG
    return causal, enc_mask


@pytest.mark.parametrize("kind", ["self", "cross", "block", "stack"])
def test_closer_to_fp32_than_hf_under_autocast(kind):
    d, H, d_ff = 512, 8, 1056
    stack = _hf_stack(d, H, d_ff, 3)
    w, blocks64, final64 = _weights(stack)
    cu_q, cuq = _cu(LQ)
    cu_k, cuk = _cu(LK)
    T, L = max(LQ), max(LK)
    x = _rows(LQ, d, 21)
    enc = _rows(LK, d, 22, torch.float32)  # the aligner's fp32 output (bf16 values, so HF's cast and ours see the same numbers)
    dy = _rows(LQ, d, 23)
    causal, enc_mask = _hf_masks(LQ, LK)
    xp, ep = _pad(x, cu_q, T).requires_grad_(True), _pad(enc, cu_k, L).requires_grad_(True)
    blk = stack.block[0]
    with torch.autocast("cuda", dtype=torch.bfloat16):
        if kind == "self":
            want = blk.layer[0](xp, attention_mask=causal)[0]
        elif kind == "cross":
            want = blk.layer[1](xp, key_value_states=ep, attention_mask=enc_mask)[0]
        elif kind == "block":
            want = blk(xp, attention_mask=causal, encoder_hidden_states=ep, encoder_attention_mask=enc_mask)[0]
        else:
            mask01 = (enc_mask[:, 0, 0] == 0).long()
            want = stack(inputs_embeds=xp, encoder_hidden_states=ep, encoder_attention_mask=mask01).last_hidden_state
    want.backward(_pad(dy, cu_q, T).to(want.dtype))
    xk, ek = x.clone().requires_grad_(True), enc.clone().requires_grad_(True)
    bias = w.position_bias
    if kind == "self":
        got = td.t5_layer_self_attention(xk, cuq, T, w.blocks[0], bias)
        fn = lambda xr, er: ref.self_attention_layer(xr, blocks64[0], cu_q, H, _bias64(w), EPS)  # noqa: E731
    elif kind == "cross":
        got = td.t5_layer_cross_attention(xk, ek, cuq, cuk, T, L, w.blocks[0])
        fn = lambda xr, er: ref.cross_attention_layer(xr, er, blocks64[0], cu_q, cu_k, H, EPS)  # noqa: E731
    elif kind == "block":
        got = td.t5_decoder_block(xk, ek, cuq, cuk, T, L, w.blocks[0], bias)
        fn = lambda xr, er: ref.block(xr, er, blocks64[0], cu_q, cu_k, H, _bias64(w), EPS)  # noqa: E731
    else:
        got = td.t5_decoder_stack(xk, ek, cuq, cuk, T, L, w)
        fn = lambda xr, er: ref.stack(xr, er, blocks64, final64, cu_q, cu_k, H, _bias64(w), EPS)  # noqa: E731
    got.backward(dy)
    r_out, r_dx, r_denc = ref.with_grads(fn, x, None if kind == "self" else enc, dy)
    hf_out = _unpad(want.detach(), cu_q)
    errs = {"out": (_rel(got, r_out), _rel(hf_out, r_out)), "dx": (_rel(xk.grad, r_dx), _rel(_unpad(xp.grad, cu_q), r_dx))}
    if kind != "self":
        assert ek.grad.dtype == torch.float32
        errs["d_enc"] = (_rel(ek.grad, r_denc), _rel(_unpad(ep.grad, cu_k), r_denc))
        assert all(not ep.grad[b, n:].any() for b, n in enumerate(LK))
    for name in ("out", "d_enc"):
        if name in errs:
            assert errs[name][0] <= 1.25 * errs[name][1], errs
    assert errs["dx"][0] <= max(1e-2, 1.25 * errs["dx"][1]), errs


def test_stack_lm_head_cross_entropy_end_to_end_vs_hf():
    d, H, d_ff, V = 512, 8, 1056, 512
    stack = _hf_stack(d, H, d_ff, 3)
    w, blocks64, final64 = _weights(stack)
    cu_q, cuq = _cu(LQ)
    cu_k, cuk = _cu(LK)
    T, L = max(LQ), max(LK)
    g = torch.Generator(device="cuda").manual_seed(31)
    w_lm = (torch.randn((V, d), generator=g, device="cuda") * d ** -0.5).to(torch.bfloat16)
    labels = torch.randint(0, V, (cu_q[-1],), generator=g, device="cuda")
    labels[torch.rand((cu_q[-1],), generator=g, device="cuda") < 0.2] = -100
    x = _rows(LQ, d, 32)
    enc = _rows(LK, d, 33, torch.float32)
    ek = enc.clone().requires_grad_(True)
    loss = td.lm_head_cross_entropy(td.t5_decoder_stack(x, ek, cuq, cuk, T, L, w), w_lm, labels)
    loss.backward()
    # HF: padded batch, encoder mask, no decoder mask (causal only), labels -100 on the pad rows
    ep = _pad(enc, cu_k, L).requires_grad_(True)
    lab_p = torch.full((len(LQ), T), -100, dtype=torch.long, device="cuda")
    for b, n in enumerate(LQ):
        lab_p[b, :n] = labels[cu_q[b] : cu_q[b + 1]]
    mask01 = torch.zeros((len(LK), L), dtype=torch.long, device="cuda")
    for b, n in enumerate(LK):
        mask01[b, :n] = 1
    head = torch.nn.Linear(d, V, bias=False, device="cuda", dtype=torch.bfloat16).requires_grad_(False)
    with torch.no_grad():
        head.weight.copy_(w_lm)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        seq = stack(inputs_embeds=_pad(x, cu_q, T), encoder_hidden_states=ep, encoder_attention_mask=mask01).last_hidden_state
        hf_loss = torch.nn.functional.cross_entropy(head(seq).view(-1, V), lab_p.view(-1), ignore_index=-100)
    hf_loss.backward()
    er = enc.double().requires_grad_(True)
    r_seq = ref.stack(x.double(), er, blocks64, final64, cu_q, cu_k, H, _bias64(w), EPS)
    r_loss = torch.nn.functional.cross_entropy(r_seq @ w_lm.double().t(), labels, ignore_index=-100)
    r_loss.backward()
    loss_err, hf_loss_err = abs(float(loss) - float(r_loss)), abs(float(hf_loss) - float(r_loss))
    # a scalar's error is one draw of the rounding noise: the 1.25x rule gets a floor of 1e-4 of the loss
    assert loss_err <= 1.25 * hf_loss_err + 1e-4 * abs(float(r_loss)), (loss_err, hf_loss_err, float(r_loss))
    assert _rel(ek.grad, er.grad) <= 1.25 * _rel(_unpad(ep.grad, cu_k), er.grad), (_rel(ek.grad, er.grad), _rel(_unpad(ep.grad, cu_k), er.grad))


def test_fp32_enc_gradient_is_summed_in_fp32():
    d, H, d_ff = 512, 8, 1056
    w, blocks64, final64 = _weights(_hf_stack(d, H, d_ff, 3))
    cu_q, cuq = _cu(LQ)
    cu_k, cuk = _cu(LK)
    T, L = max(LQ), max(LK)
    x, dy = _rows(LQ, d, 41), _rows(LQ, d, 42)
    enc = _rows(LK, d, 43, torch.float32)
    e32, e16 = enc.clone().requires_grad_(True), enc.to(torch.bfloat16).requires_grad_(True)
    for e in (e32, e16):
        td.t5_decoder_stack(x, e, cuq, cuk, T, L, w).backward(dy)
    _, _, r_denc = ref.with_grads(lambda xr, er: ref.stack(xr, er, blocks64, final64, cu_q, cu_k, H, _bias64(w), EPS), x, enc, dy)
    assert e32.grad.dtype == torch.float32 and e16.grad.dtype == torch.bfloat16
    assert not torch.equal(e32.grad.to(torch.bfloat16).float(), e32.grad)  # not rounded to bf16 anywhere on the way
    assert _rel(e32.grad, r_denc) < _rel(e16.grad, r_denc)


def test_bit_identical_across_runs_and_inference_path():
    d, H = 4096, 64
    stack = _hf_stack(d, H, 1024, 1)
    w, _, _ = _weights(stack)
    lens_q, lens_k = _lens("cfg", "cfg", seed=8)
    cu_q, cuq = _cu(lens_q)
    cu_k, cuk = _cu(lens_k)
    T, L = max(lens_q), max(lens_k)
    x, dy = _rows(lens_q, d, 51), _rows(lens_q, d, 52)
    enc = _rows(lens_k, d, 53, torch.float32)
    runs = []
    for _ in range(2):
        xk, ek = x.clone().requires_grad_(True), enc.clone().requires_grad_(True)
        out = td.t5_decoder_block(xk, ek, cuq, cuk, T, L, w.blocks[0], w.position_bias)
        out.backward(dy)
        runs.append((out.detach(), xk.grad, ek.grad))
    for t0, t1 in zip(*runs):
        assert torch.equal(t0, t1)
    with torch.no_grad():
        assert torch.equal(td.t5_decoder_block(x, enc, cuq, cuk, T, L, w.blocks[0], w.position_bias), runs[0][0])
    bw = w.blocks[0]
    o_train = ops.t5_self_attention_layer_fwd(x, bw.w_qkv, bw.wo_self, bw.ln_self, EPS, w.position_bias, cuq, T, H)
    o_inf = ops.t5_self_attention_layer_fwd(x, bw.w_qkv, bw.wo_self, bw.ln_self, EPS, w.position_bias, cuq, T, H, want_saved=False)
    assert all(t is None for t in o_inf[1:]) and torch.equal(o_train[0], o_inf[0])
    e16 = enc.to(torch.bfloat16)
    c_train = ops.t5_cross_attention_layer_fwd(x, e16, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, EPS, cuq, cuk, T, L, H)
    c_inf = ops.t5_cross_attention_layer_fwd(x, e16, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, EPS, cuq, cuk, T, L, H, want_saved=False)
    assert all(t is None for t in c_inf[1:]) and torch.equal(c_train[0], c_inf[0])


def test_empty_batch_is_a_no_op():
    w, _, _ = _weights(_hf_stack(512, 8, 1024, 1))
    bw = w.blocks[0]
    x = torch.empty((0, 512), dtype=torch.bfloat16, device="cuda")
    cu = torch.zeros((1,), dtype=torch.int32, device="cuda")
    out, rstd, qkv, o, lse = ops.t5_self_attention_layer_fwd(x, bw.w_qkv, bw.wo_self, bw.ln_self, EPS, w.position_bias, cu, 0, 8)
    dx, _ = ops.t5_self_attention_layer_bwd(x, x, rstd, qkv, o, lse, bw.w_qkv, bw.wo_self, bw.ln_self, w.position_bias, cu, 0, 8)
    assert out.shape == (0, 512) and dx.shape == (0, 512)
    enc = torch.empty((0, 512), dtype=torch.bfloat16, device="cuda")
    out, rstd, q, kv, o, lse = ops.t5_cross_attention_layer_fwd(x, enc, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, EPS, cu, cu, 0, 0, 8)
    dx, d_enc = ops.t5_cross_attention_layer_bwd(x, x, rstd, q, kv, o, lse, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, cu, cu, 0, 0, 8)
    assert out.shape == (0, 512) and d_enc.shape == (0, 512)
    lib = _lib.lib()
    assert lib.td_t5_self_attention_layer_fwd(None, 0, 512, 8, None, 0, 0, None, EPS, None, None, None, 0, None, None, None, None, None,
                                              None, 0, None) == 0
    assert lib.td_t5_cross_attention_layer_bwd(*([None] * 13), 0, 0, 0, 0, 0, 512, 8, None, None, None, 0, None) == 0
    # decoder rows whose samples have no aligner rows at all: out = x, d_enc empty
    cu_q, cuq = _cu([3, 5])
    xs, dys = _rows([3, 5], 512, 61), _rows([3, 5], 512, 62)
    cuk = torch.zeros((3,), dtype=torch.int32, device="cuda")
    out, rstd, q, kv, o, lse = ops.t5_cross_attention_layer_fwd(xs, enc, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, EPS, cuq, cuk, 5, 0, 8)
    assert torch.equal(out, xs)
    dx, d_enc = ops.t5_cross_attention_layer_bwd(dys, xs, rstd, q, kv, o, lse, bw.w_q, bw.w_kv, bw.wo_cross, bw.ln_cross, cuq, cuk, 5, 0, 8)
    assert d_enc.shape == (0, 512) and bool(torch.isfinite(dx.float()).all())


def test_rejected_arguments():
    lib = _lib.lib()
    w, _, _ = _weights(_hf_stack(512, 8, 1024, 1))
    bw = w.blocks[0]
    M, d, H = 64, 512, 8
    cu_q, cuq = _cu([M])
    x = _rows([M], d, 71)
    out = torch.empty_like(x)
    ws_bytes = lib.td_t5_attention_layer_workspace_bytes(M, 0, d, H, 1)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    P, s = _lib.ptr, _lib.stream_ptr()

    def fwd(x_, d_=d, H_=H, bias=w.position_bias, ws_bytes_=ws_bytes, w_qkv=bw.w_qkv):
        return lib.td_t5_self_attention_layer_fwd(P(x_), M, d_, H_, P(cuq), 1, M, P(bw.ln_self), EPS, P(w_qkv), P(bw.wo_self), P(bias),
                                                  128, P(out), None, None, None, None, P(ws), ws_bytes_, s)

    assert fwd(x) == 0
    assert fwd(x, d_=480) != 0 and "d %" in _lib.last_error()
    assert fwd(x, d_=8192) != 0 and "d <=" in _lib.last_error()
    assert fwd(x, H_=0) != 0 and "bad sizes" in _lib.last_error()
    assert fwd(x, ws_bytes_=ws_bytes - 256) != 0 and "workspace" in _lib.last_error()
    assert fwd(x, bias=None) != 0 and "relative position bias" in _lib.last_error()
    buf = torch.empty((M * d + 8,), dtype=torch.bfloat16, device="cuda")
    assert fwd(buf[1 : 1 + M * d].view(M, d)) != 0 and "aligned" in _lib.last_error()
    assert fwd(x, w_qkv=None) != 0 and "null pointer" in _lib.last_error()
    with pytest.raises(RuntimeError, match="td_t5_self_attention_layer_bwd"):  # the backward needs the forward's lse
        lib_rc = lib.td_t5_self_attention_layer_bwd(P(x), P(x), P(x), P(bw.ln_self), P(x), P(x), None, P(bw.w_qkv), P(bw.wo_self),
                                                    P(w.position_bias), 128, P(cuq), 1, M, M, d, H, P(out), None, P(ws), ws_bytes, s)
        _lib.check(lib_rc, "td_t5_self_attention_layer_bwd")
    assert "null pointer" in _lib.last_error()
    with pytest.raises(TypeError, match="w_qkv"):
        ops.t5_self_attention_layer_fwd(x, bw.w_qkv[: 3 * 64 * 4], bw.wo_self, bw.ln_self, EPS, w.position_bias, cuq, M, H)
    with pytest.raises(TypeError, match="want_saved=True"):
        o = ops.t5_self_attention_layer_fwd(x, bw.w_qkv, bw.wo_self, bw.ln_self, EPS, w.position_bias, cuq, M, H, want_saved=False)
        ops.t5_self_attention_layer_bwd(x, x, *o[1:], bw.w_qkv, bw.wo_self, bw.ln_self, w.position_bias, cuq, M, H)
    enc = _rows([5], d, 72)
    cuk = torch.tensor([0, 5], dtype=torch.int32, device="cuda")
    cws = lib.td_t5_attention_layer_workspace_bytes(M, 5, d, H, 0)
    ws2 = torch.empty((cws,), dtype=torch.uint8, device="cuda")
    rc = lib.td_t5_cross_attention_layer_fwd(P(x), M, P(enc), 5, d, H, P(cuq), None, 1, M, 5, P(bw.ln_cross), EPS, P(bw.w_q), P(bw.w_kv),
                                             P(bw.wo_cross), P(out), None, None, None, None, None, P(ws2), cws, s)
    assert rc != 0 and "null pointer" in _lib.last_error()  # cross-attention needs cu_k
    rc = lib.td_t5_cross_attention_layer_fwd(P(x), M, P(enc), 5, d, H, P(cuq), P(cuk), 1, M, 5, P(bw.ln_cross), EPS, P(bw.w_q), P(bw.w_kv),
                                             P(bw.wo_cross), P(out), None, None, None, None, None, P(ws2), cws - 256, s)
    assert rc != 0 and "workspace" in _lib.last_error()
    with pytest.raises(NotImplementedError, match="require grad"):
        td.T5DecoderBlockWeights(bw.ln_self.clone().requires_grad_(True), *([bw.w_q.float()] * 3), bw.wo_self, bw.ln_cross,
                                 *([bw.w_q] * 3), bw.wo_cross, bw.ffn, H)
