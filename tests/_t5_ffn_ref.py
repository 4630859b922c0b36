"""Reference of the T5 gated-GELU feed-forward sublayer (``T5LayerFF`` with ``T5DenseGatedActDense``) -- test infrastructure only, the
product path never imports it. tests/test_t5_ffn_cpu.py pins ``layer_ff`` live to transformers' ``T5LayerFF``; tests/test_gpu_t5_ffn.py
compares the kernels against it, and against the "staged" functions, which apply the kernels' bf16 rounding points to given
intermediates (header include/thinkdiff_b200.h, td_t5_ffn_fwd)."""
from __future__ import annotations

import math

import torch

_C = math.sqrt(2.0 / math.pi)


def gelu_new(x: torch.Tensor) -> torch.Tensor:
    """transformers' NewGELUActivation (the tanh form), in x's dtype."""
    return 0.5 * x * (1.0 + torch.tanh(_C * (x + 0.044715 * x.pow(3))))


def gelu_new_grad(x: torch.Tensor) -> torch.Tensor:
    t = torch.tanh(_C * (x + 0.044715 * x.pow(3)))
    return 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * _C * (1.0 + 3 * 0.044715 * x * x)


def layer_ff(x, ln_w, wi_0, wi_1, wo, eps: float):
    """``x + wo(gelu_new(wi_0(norm(x))) * wi_1(norm(x)))`` with T5's RMSNorm, everything in x's dtype (float32 / float64)."""
    xn = ln_w * (x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + eps))
    return x + (gelu_new(xn @ wi_0.t()) * (xn @ wi_1.t())) @ wo.t()


def layer_ff_with_grad(x, ln_w, wi_0, wi_1, wo, eps: float, dy, dtype=torch.float64):
    """(out, dx) of ``layer_ff`` in ``dtype`` from the given (e.g. bf16) tensors; dx = the gradient of (out * dy).sum() to x."""
    xr = x.detach().to(dtype).requires_grad_(True)
    out = layer_ff(xr, *(t.detach().to(dtype) for t in (ln_w, wi_0, wi_1, wo)), eps)
    out.backward(dy.to(dtype))
    return out.detach(), xr.grad


def _bf(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(t.dtype)


def gated_staged(a: torch.Tensor, b: torch.Tensor, nudge: float = 1.0) -> torch.Tensor:
    """g = bf16(bf16(gelu_new(a)) * b) from bf16 a, b; gelu_new evaluated in float64 (and multiplied by ``nudge`` before rounding)."""
    a, b = a.double(), b.double()
    return (_bf(gelu_new(a) * nudge) * b).to(torch.bfloat16)


def dgated_staged(t: torch.Tensor, a: torch.Tensor, b: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """(d_a, d_b) from t = dy . wo (any precision, rounded to bf16 here) and bf16 a, b:
    d_a = bf16(bf16(t * b) * gelu_new'(a)), d_b = bf16(t * bf16(gelu_new(a)))."""
    t, a, b = _bf(t.double()), a.double(), b.double()
    d_b = (t * _bf(gelu_new(a))).to(torch.bfloat16)
    d_a = (_bf(t * b) * gelu_new_grad(a)).to(torch.bfloat16)
    return d_a, d_b
