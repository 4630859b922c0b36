"""CPU checks of the T5 gated-GELU FFN sublayer's host side: the weight interleave and its inverse, the frozen weight holder built
from a live transformers ``T5LayerFF``, the reference pinned to HF, the workspace size function, and the work schedules of the three
new GEMM shapes (the property checks of test_gemm_schedule.py, run on them)."""
import pytest
import torch

import _t5_ffn_ref as ref
from test_gemm_schedule import test_every_k_block_of_every_tile_is_computed_exactly_once as _every_k_block_once
from test_gemm_schedule import test_shared_tiles_have_one_owner_whose_contributors_are_claimed_first as _owner_and_contributors
from thinkdiff_mlre_b200 import _lib
from thinkdiff_mlre_b200.t5 import T5FeedForwardWeights, interleave_pairs, split_pairs


def _hf_layer(d, d_ff, seed=0):
    transformers = pytest.importorskip("transformers")
    from transformers.models.t5.modeling_t5 import T5LayerFF

    torch.manual_seed(seed)
    cfg = transformers.T5Config(d_model=d, d_ff=d_ff, feed_forward_proj="gated-gelu", dropout_rate=0.0)
    layer = T5LayerFF(cfg).eval()
    with torch.no_grad():
        layer.layer_norm.weight.copy_(1.0 + 0.1 * torch.randn(d))
    return layer


@pytest.mark.parametrize("d_ff", [32, 96, 1024, 1056])
def test_interleave_round_trip_and_layout(d_ff):
    d = 64
    w0, w1 = torch.randn(d_ff, d), torch.randn(d_ff, d)
    wi = interleave_pairs(w0, w1)
    assert wi.shape == (2 * d_ff, d)
    for k in range(d_ff // 32):
        assert torch.equal(wi[64 * k : 64 * k + 32], w0[32 * k : 32 * k + 32])
        assert torch.equal(wi[64 * k + 32 : 64 * k + 64], w1[32 * k : 32 * k + 32])
    a, b = split_pairs(wi)
    assert torch.equal(a, w0) and torch.equal(b, w1)
    # along columns: what ab = xn . wi^T looks like, and its inverse gives xn . wi_0^T, xn . wi_1^T
    xn = torch.randn(5, d)
    a, b = split_pairs(xn @ wi.t(), dim=1)
    assert torch.allclose(a, xn @ w0.t()) and torch.allclose(b, xn @ w1.t())
    assert torch.equal(interleave_pairs(a, b, dim=1), xn @ wi.t())
    with pytest.raises(ValueError):
        interleave_pairs(torch.randn(48, d), torch.randn(48, d))
    with pytest.raises(ValueError):
        split_pairs(torch.randn(96, d))


def test_weights_from_a_live_hf_layer_and_its_state_dict():
    layer = _hf_layer(128, 96)
    with pytest.raises(NotImplementedError, match="require grad"):
        T5FeedForwardWeights.from_module(layer)
    layer.requires_grad_(False)
    w = T5FeedForwardWeights.from_module(layer)
    ff = layer.DenseReluDense
    assert (w.d, w.d_ff, w.eps) == (128, 96, layer.layer_norm.variance_epsilon)
    assert w.wi.dtype == torch.bfloat16 and w.wo.dtype == torch.bfloat16 and w.ln_weight.dtype == torch.float32
    a, b = T5FeedForwardWeights.split(w.wi)
    assert torch.equal(a, ff.wi_0.weight.to(torch.bfloat16)) and torch.equal(b, ff.wi_1.weight.to(torch.bfloat16))
    assert torch.equal(w.wo, ff.wo.weight.to(torch.bfloat16)) and torch.equal(w.ln_weight, layer.layer_norm.weight)
    w2 = T5FeedForwardWeights.from_state_dict({"layer.1." + k: v for k, v in layer.state_dict().items()}, prefix="layer.1.")
    assert torch.equal(w2.wi, w.wi) and torch.equal(w2.wo, w.wo) and torch.equal(w2.ln_weight, w.ln_weight)
    with pytest.raises(ValueError):
        T5FeedForwardWeights(ff.wi_0.weight, ff.wi_1.weight[:64], ff.wo.weight, layer.layer_norm.weight)


def test_reference_equals_hf_t5_layer_ff_in_fp32():
    layer = _hf_layer(128, 192, seed=1)
    ff = layer.DenseReluDense
    torch.manual_seed(2)
    x = torch.randn(37, 128, requires_grad=True)
    dy = torch.randn(37, 128)
    out = layer(x)
    out.backward(dy)
    r_out, r_dx = ref.layer_ff_with_grad(x, layer.layer_norm.weight, ff.wi_0.weight, ff.wi_1.weight, ff.wo.weight,
                                         layer.layer_norm.variance_epsilon, dy, dtype=torch.float32)
    assert (r_out - out.detach()).abs().max() <= 1e-5
    assert (r_dx - x.grad).abs().max() <= 1e-5
    # the closed-form derivative the staged backward uses
    z = torch.linspace(-8, 8, 2001, dtype=torch.float64, requires_grad=True)
    ref.gelu_new(z).sum().backward()
    assert (z.grad - ref.gelu_new_grad(z.detach())).abs().max() <= 1e-12


def test_ffn_workspace_size_is_pure_aligned_and_monotone():
    f = _lib.lib().td_t5_ffn_workspace_bytes
    prev = 0
    for m in (0, 1, 127, 128, 1000, 4352, 8192):
        n = f(m, 4096, 10240)
        assert n == f(m, 4096, 10240) and n % 256 == 0 and n >= prev
        assert n >= 2 * max(m, 1) * (4096 + 2 * 10240)  # the [M, d] and [M, 2 d_ff] bf16 buffers
        prev = n
    assert f(1000, 512, 1056) < f(1000, 4096, 10240)


D, D_FF = 4096, 10240
FFN_SHAPES = {"gate": lambda m: (m, 2 * D_FF, D), "dgate": lambda m: (m, D_FF, D), "dx": lambda m: (m, D, 2 * D_FF)}


@pytest.mark.parametrize("M", [1, 129, 1000, 4352, 8192])
@pytest.mark.parametrize("gemm", sorted(FFN_SHAPES))
def test_ffn_gemm_schedules(gemm, M):
    shape = FFN_SHAPES[gemm](M)
    _every_k_block_once(shape, 74)
    _owner_and_contributors(shape, 74)
