"""CPU checks of the T5 decoder block's host side: the float64 packed-row references of tests/_t5_decoder_block_ref.py pinned live to
transformers' ``T5LayerSelfAttention``, ``T5LayerCrossAttention`` and ``T5Block`` (fp32, zero-padded batch + masks, ragged decoder and
aligner lengths: outputs, and the gradients into the decoder rows and the aligner rows, with exactly none on HF's pad rows); the frozen
weight holders built from a live ``T5Block`` / ``T5Stack`` and from their state dicts; the attention sublayers' workspace size
function; and the work schedules of the new GEMM shapes at the cfg2 / cfg5 row counts."""
import pytest
import torch

import _t5_decoder_block_ref as ref
from test_gemm_schedule import test_every_k_block_of_every_tile_is_computed_exactly_once as _every_k_block_once
from test_gemm_schedule import test_shared_tiles_have_one_owner_whose_contributors_are_claimed_first as _owner_and_contributors
from thinkdiff_mlre_b200 import _lib
from thinkdiff_mlre_b200.t5 import T5DecoderBlockWeights, T5DecoderWeights, T5FeedForwardWeights, t5_position_bias_by_distance

transformers = pytest.importorskip("transformers")
D, H, D_FF, EPS = 128, 2, 96, 1e-6
NEG = torch.finfo(torch.float32).min


def _cfg(n_layers=1, d_kv=64):
    return transformers.T5Config(vocab_size=32, d_model=D, d_kv=d_kv, d_ff=D_FF, num_layers=n_layers, num_decoder_layers=n_layers, num_heads=H,
                                 relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                                 feed_forward_proj="gated-gelu", is_decoder=True, use_cache=False, layer_norm_epsilon=EPS)


def _randomize(module, seed):
    torch.manual_seed(seed)
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(1.0 + 0.1 * torch.randn(p.shape) if p.dim() == 1 else torch.randn(p.shape) * 0.5 * p.shape[-1] ** -0.5)
    return module.eval()


def _cu(lens):
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    return cu


def _pad(x, cu, L):
    out = x.new_zeros((len(cu) - 1, L, x.shape[1]))
    for b in range(len(cu) - 1):
        out[b, : cu[b + 1] - cu[b]] = x[cu[b] : cu[b + 1]]
    return out


def _unpad(xp, cu):
    return torch.cat([xp[b, : cu[b + 1] - cu[b]] for b in range(len(cu) - 1)])


def _masks(lens_q, lens_k):
    T, L = max(lens_q), max(lens_k)
    causal = torch.full((T, T), NEG).triu(1)[None, None].expand(len(lens_q), 1, T, T)
    enc_mask = torch.zeros((len(lens_k), 1, 1, L))
    for b, n in enumerate(lens_k):
        enc_mask[b, ..., n:] = NEG
    return causal, enc_mask


def _inputs(lens_q, lens_k, seed):
    g = torch.Generator().manual_seed(seed)
    cu_q, cu_k = _cu(lens_q), _cu(lens_k)
    x = torch.randn((cu_q[-1], D), generator=g)
    enc = torch.randn((cu_k[-1], D), generator=g)
    up = torch.randn((cu_q[-1], D), generator=g)
    return cu_q, cu_k, x, enc, up


def _check(got, want, atol):
    assert float((got.double() - want.double()).abs().max()) <= atol * (1.0 + float(want.abs().max()))


LENS = [([5, 1, 17, 9], [7, 3, 40, 1]), ([1], [1]), ([33, 12], [2, 130])]


@pytest.mark.parametrize("lens_q,lens_k", LENS)
@pytest.mark.parametrize("kind", ["self", "cross", "block"])
def test_reference_equals_hf_on_the_padded_batch(kind, lens_q, lens_k):
    from transformers.models.t5.modeling_t5 import T5Block, T5LayerCrossAttention, T5LayerSelfAttention

    cu_q, cu_k, x, enc, up = _inputs(lens_q, lens_k, seed=sum(lens_q) + len(kind))
    T, L = max(lens_q), max(lens_k)
    causal, enc_mask = _masks(lens_q, lens_k)
    xp, ep = _pad(x, cu_q, T).requires_grad_(True), _pad(enc, cu_k, L).requires_grad_(True)
    if kind == "self":
        layer = _randomize(T5LayerSelfAttention(_cfg(), has_relative_attention_bias=True, layer_idx=0), 1)
        want = layer(xp, attention_mask=causal)[0]
        w = {"layer.0." + k: v for k, v in layer.state_dict().items()}
        table = layer.SelfAttention.relative_attention_bias.weight
    elif kind == "cross":
        layer = _randomize(T5LayerCrossAttention(_cfg(), layer_idx=0), 2)
        want = layer(xp, key_value_states=ep, attention_mask=enc_mask)[0]
        w = {"layer.1." + k: v for k, v in layer.state_dict().items()}
        table = None
    else:
        layer = _randomize(T5Block(_cfg(), has_relative_attention_bias=True, layer_idx=0), 3)
        want = layer(xp, attention_mask=causal, encoder_hidden_states=ep, encoder_attention_mask=enc_mask)[0]
        w = layer.state_dict()
        table = layer.layer[0].SelfAttention.relative_attention_bias.weight
    want.backward(_pad(up, cu_q, T))
    bias = None if table is None else t5_position_bias_by_distance(table.detach()).double()
    w64 = ref.to(w, torch.float64)
    fn = {
        "self": lambda xr, er: ref.self_attention_layer(xr, w64, cu_q, H, bias, EPS),
        "cross": lambda xr, er: ref.cross_attention_layer(xr, er, w64, cu_q, cu_k, H, EPS),
        "block": lambda xr, er: ref.block(xr, er, w64, cu_q, cu_k, H, bias, EPS),
    }[kind]
    r_out, r_dx, r_denc = ref.with_grads(fn, x, None if kind == "self" else enc, up)
    _check(r_out, _unpad(want.detach(), cu_q), 1e-5)
    _check(r_dx, _unpad(xp.grad, cu_q), 1e-5)
    assert all(not xp.grad[b, n:].any() for b, n in enumerate(lens_q))  # HF's decoder pad rows: exactly no gradient
    if kind != "self":
        _check(r_denc, _unpad(ep.grad, cu_k), 1e-5)
        assert all(not ep.grad[b, n:].any() for b, n in enumerate(lens_k))  # masked aligner rows: exactly no gradient


def test_cross_reference_sample_without_aligner_rows_passes_x_through():
    cu_q, cu_k, x, enc, up = _inputs([4, 6], [0, 5], seed=9)
    layer = _randomize(transformers.models.t5.modeling_t5.T5LayerCrossAttention(_cfg(), layer_idx=0), 4)
    w64 = ref.to({"layer.1." + k: v for k, v in layer.state_dict().items()}, torch.float64)
    out, dx, d_enc = ref.with_grads(lambda xr, er: ref.cross_attention_layer(xr, er, w64, cu_q, cu_k, H, EPS), x, enc, up)
    assert torch.equal(out[:4], x[:4].double()) and torch.equal(dx[:4], up[:4].double())
    assert d_enc.shape == enc.shape and d_enc.abs().sum() > 0


def _block(seed=0, d_kv=64):
    from transformers.models.t5.modeling_t5 import T5Block

    return _randomize(T5Block(_cfg(d_kv=d_kv), has_relative_attention_bias=True, layer_idx=0), seed)


def _assert_block_weights(w, blk):
    sa, ca = blk.layer[0].SelfAttention, blk.layer[1].EncDecAttention
    bf = torch.bfloat16
    assert (w.d, w.n_heads, w.eps) == (D, H, EPS)
    assert torch.equal(w.w_qkv, torch.cat([sa.q.weight, sa.k.weight, sa.v.weight]).to(bf)) and torch.equal(w.wo_self, sa.o.weight.to(bf))
    assert torch.equal(w.w_q, ca.q.weight.to(bf)) and torch.equal(w.w_kv, torch.cat([ca.k.weight, ca.v.weight]).to(bf))
    assert torch.equal(w.wo_cross, ca.o.weight.to(bf))
    assert w.ln_self.dtype == torch.float32 and torch.equal(w.ln_self, blk.layer[0].layer_norm.weight)
    assert torch.equal(w.ln_cross, blk.layer[1].layer_norm.weight)
    a, b = T5FeedForwardWeights.split(w.ffn.wi)
    assert torch.equal(a, blk.layer[2].DenseReluDense.wi_0.weight.to(bf)) and torch.equal(b, blk.layer[2].DenseReluDense.wi_1.weight.to(bf))
    for t in (w.w_qkv, w.wo_self, w.w_q, w.w_kv, w.wo_cross):
        assert t.dtype == bf and t.is_contiguous()


def test_block_weights_from_a_live_t5_block_and_its_state_dict():
    blk = _block()
    with pytest.raises(NotImplementedError, match="require grad"):
        T5DecoderBlockWeights.from_module(blk)
    blk.requires_grad_(False)
    w = T5DecoderBlockWeights.from_module(blk)
    _assert_block_weights(w, blk)
    w2 = T5DecoderBlockWeights.from_state_dict({"decoder.block.0." + k: v for k, v in blk.state_dict().items()}, n_heads=H, eps=EPS,
                                               prefix="decoder.block.0.")
    _assert_block_weights(w2, blk)
    with pytest.raises(NotImplementedError, match="d_kv"):
        T5DecoderBlockWeights.from_state_dict(blk.state_dict(), n_heads=4)  # 128-wide projections over 4 heads: d_kv = 32


def test_block_weights_refuse_d_kv_other_than_64():
    blk = _block(d_kv=32).requires_grad_(False)
    with pytest.raises(NotImplementedError, match="d_kv"):
        T5DecoderBlockWeights.from_module(blk)


def test_decoder_weights_from_a_live_t5_stack_and_its_state_dict():
    from transformers.models.t5.modeling_t5 import T5Stack

    stack = _randomize(T5Stack(_cfg(n_layers=3)), 5)
    with pytest.raises(NotImplementedError, match="require grad"):
        T5DecoderWeights.from_module(stack)
    stack.requires_grad_(False)
    w = T5DecoderWeights.from_module(stack)
    table = stack.block[0].layer[0].SelfAttention.relative_attention_bias.weight
    assert len(w.blocks) == 3 and w.eps == EPS
    assert torch.equal(w.position_bias, t5_position_bias_by_distance(table)) and w.position_bias.shape == (H, 128)
    assert torch.equal(w.final_ln, stack.final_layer_norm.weight)
    for wb, blk in zip(w.blocks, stack.block):
        _assert_block_weights(wb, blk)
    w2 = T5DecoderWeights.from_state_dict({"decoder." + k: v for k, v in stack.state_dict().items()}, n_heads=H, eps=EPS, prefix="decoder.")
    assert len(w2.blocks) == 3 and torch.equal(w2.position_bias, w.position_bias) and torch.equal(w2.final_ln, w.final_ln)
    for wb, blk in zip(w2.blocks, stack.block):
        _assert_block_weights(wb, blk)


def test_attention_layer_workspace_size_is_pure_aligned_and_monotone():
    f = _lib.lib().td_t5_attention_layer_workspace_bytes
    d, h = 4096, 64
    inner = 64 * h
    for self_attention in (1, 0):
        prev = 0
        for m in (0, 1, 127, 128, 4506, 8217):
            for mk in (0, 1, 7474, 63698):
                n = f(m, mk, d, h, self_attention)
                assert n == f(m, mk, d, h, self_attention) and n % 256 == 0
                rows = max(m, 1)
                proj = 3 * rows * inner if self_attention else 2 * max(mk, 1) * inner + rows * inner
                assert n >= 2 * (rows * d + proj + rows * inner) + 4 * rows * (1 + h)  # xn, qkv | q + kv, o, rstd, delta
                assert n >= f(m, 0, d, h, self_attention)
            assert f(m, 7474, d, h, self_attention) >= prev
            prev = f(m, 7474, d, h, self_attention)
        assert f(1000, 7474, 512, 8, self_attention) < f(1000, 7474, 4096, 64, self_attention)
    assert f(4506, 123, d, h, 1) == f(4506, 0, d, h, 1)  # self-attention ignores Mk


DM, INNER = 4096, 4096
ROWS = {"cfg2_dec": 4506, "cfg5_dec": 8217, "cfg2_enc": 7474, "cfg5_enc": 63698}
LAYER_SHAPES = {  # (rows, N, K) of every GEMM of the two sublayers
    "sa_qkv": ("dec", 3 * INNER, DM), "sa_out": ("dec", DM, INNER), "sa_do": ("dec", INNER, DM), "sa_dx": ("dec", DM, 3 * INNER),
    "ca_q": ("dec", INNER, DM), "ca_kv": ("enc", 2 * INNER, DM), "ca_dq": ("dec", DM, INNER), "ca_denc": ("enc", DM, 2 * INNER),
}


@pytest.mark.parametrize("cfg", ["cfg2", "cfg5"])
@pytest.mark.parametrize("gemm", sorted(LAYER_SHAPES))
def test_attention_layer_gemm_schedules(gemm, cfg):
    rows, N, K = LAYER_SHAPES[gemm]
    shape = (ROWS[f"{cfg}_{rows}"], N, K)
    _every_k_block_once(shape, 74)
    _owner_and_contributors(shape, 74)
