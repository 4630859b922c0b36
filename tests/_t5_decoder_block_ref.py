"""Float64 references of the T5 decoder's attention sublayers, block and stack on PACKED rows -- test infrastructure only, the product
path never imports it. Built from ``_t5_attention_ref.attention_packed`` and ``_t5_ffn_ref.layer_ff``. attention_packed evaluates the
attention core in fp32 (about 1e-7 relative, far below the bf16 errors the tests measure) and runs here on the CPU, so the
projections may run on the GPU. tests/test_t5_decoder_block_cpu.py pins the references live to transformers' ``T5LayerSelfAttention``,
``T5LayerCrossAttention`` and ``T5Block`` on the zero-padded batch + masks; tests/test_gpu_t5_decoder_block.py compares the kernels
against them.

Weights come as a dict in ``T5Block`` state-dict naming without the block prefix (``layer.0.SelfAttention.q.weight``, ...)."""
from __future__ import annotations

import torch

import _t5_attention_ref
import _t5_ffn_ref


def rms_norm(x, w, eps: float):
    return w * (x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + eps))


def self_attention_layer(x, w: dict, cu_q, n_heads: int, bias_by_distance, eps: float):
    """``x + o(attention(q, k, v))`` on ``norm(x)``, causal within each sample ``cu_q[b]:cu_q[b+1]``, with the per-distance bias."""
    a = "layer.0.SelfAttention."
    xn = rms_norm(x, w["layer.0.layer_norm.weight"], eps)
    q, k, v = (xn @ w[a + n + ".weight"].t() for n in "qkv")
    o = _t5_attention_ref.attention_packed(q.cpu(), k.cpu(), v.cpu(), cu_q, None, n_heads, bias_by_distance.cpu()).to(x)
    return x + o @ w[a + "o.weight"].t()


def cross_attention_layer(x, enc, w: dict, cu_q, cu_k, n_heads: int, eps: float):
    """``x + o(attention(q(norm(x)), k(enc), v(enc)))``; decoder sample b (rows ``cu_q[b]:``) sees aligner rows ``cu_k[b]:cu_k[b+1]``."""
    a = "layer.1.EncDecAttention."
    xn = rms_norm(x, w["layer.1.layer_norm.weight"], eps)
    q = xn @ w[a + "q.weight"].t()
    k, v = enc @ w[a + "k.weight"].t(), enc @ w[a + "v.weight"].t()
    o = _t5_attention_ref.attention_packed(q.cpu(), k.cpu(), v.cpu(), cu_q, cu_k, n_heads).to(x)
    return x + o @ w[a + "o.weight"].t()


def block(x, enc, w: dict, cu_q, cu_k, n_heads: int, bias_by_distance, eps: float):
    h = self_attention_layer(x, w, cu_q, n_heads, bias_by_distance, eps)
    h = cross_attention_layer(h, enc, w, cu_q, cu_k, n_heads, eps)
    f = "layer.2.DenseReluDense."
    return _t5_ffn_ref.layer_ff(h, w["layer.2.layer_norm.weight"], w[f + "wi_0.weight"], w[f + "wi_1.weight"], w[f + "wo.weight"], eps)


def stack(x, enc, blocks: list, final_ln, cu_q, cu_k, n_heads: int, bias_by_distance, eps: float):
    for w in blocks:
        x = block(x, enc, w, cu_q, cu_k, n_heads, bias_by_distance, eps)
    return rms_norm(x, final_ln, eps)


def with_grads(fn, x, enc, dy, dtype=torch.float64):
    """``(out, dx, d_enc)`` of ``fn(x, enc)`` in ``dtype`` from the given (e.g. bf16) tensors, the gradients those of ``(out * dy).sum()``;
    ``enc`` may be None (self-attention: ``d_enc`` is None)."""
    xr = x.detach().to(dtype).requires_grad_(True)
    er = None if enc is None else enc.detach().to(dtype).requires_grad_(True)
    out = fn(xr, er)
    out.backward(dy.to(dtype))
    return out.detach(), xr.grad, None if er is None else er.grad


def to(w: dict, dtype, device=None) -> dict:
    return {k: v.detach().to(device=device, dtype=dtype) for k, v in w.items()}
