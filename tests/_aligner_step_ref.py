"""Float64 staged reference of the fused aligner train step, for per-element parity at production width.

Every stage takes the kernels' own bf16 outputs of the stage before it (h0 -> h1, h1 -> h2, h2 -> dh2, dh2 -> dh0, ...), so
errors do not compound and each bound can be tight. The rounding points are those of ``oracle.aligner_ref.aligner_fwd_bwd_manual``
(bf16 regime):

    h0 = bf16(x W1^T + b1)           h1 = bf16(gelu_erf(h0))            h2 = bf16(h1 W2^T + b2)
    rstd = (mean(h2^2) + eps)^-1/2   y = g h2 rstd (fp32)                dy = 2 (y - t) / (M D)
    dh2 = bf16(T5LayerNorm backward of dy)                               dh0 = bf16(bf16(dh2 W2) gelu'(h0))
    dg = sum_rows dy h2 rstd   db2 = sum_rows dh2   db1 = sum_rows dh0   dW2 = dh2^T h1   dW1 = dh0^T x

Everything is float64 torch arithmetic on whatever device the inputs live on (the GPU at production size, the CPU in the test
that pins this file to the oracle). A GEMM stage returns its exact product and a bound on the error of an fp32-accumulated
product of the same bf16 operands (``ACC * (|A| |B|^T)``, and for the long token contractions also the running-sum term of
``contract_rows``); ``gemm_error`` turns that into a per-element error / tolerance pair through the rounding of the GEMM's
epilogue. Large products are formed in row blocks so the float64 temporaries stay small.
"""
from __future__ import annotations

import math

import torch

# fp32 accumulation of bf16 products (exact in fp32): the tensor-core sum plus the stream-K fold of a few partials stays far inside
# 2^-18 of sum |a b|
ACC = 2.0 ** -18
# relative error of the fp32 row statistics (rstd, and the fused norm's diff = g h rstd - t built from it): the GPU test checks
# rstd to 1e-6 (about 2^-20); twice that here
ROW_EPS = 2.0 ** -19
# gelu' in the dh0 epilogue comes from the Abramowitz-Stegun erf (absolute error 1.5e-7 on erf) and MUFU ex2: good to 2^-21
# absolute -- not relative: gelu'(x) crosses zero at x = -0.75
GELU_GRAD_ABS = 2.0 ** -21
# fp32 ulp of the running sum (2^-23 |S|) for each of the four 16-deep MMA accumulations of a 64-deep k-block
RUN_SUM = 4 * 2.0 ** -23
KBLOCK = 64
BLOCK_ROWS = 2048


def bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 through fp32 (the oracle's rounding: float64 result -> float32 tensor -> bf16), returned as float64."""
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def ulp(v: torch.Tensor) -> torch.Tensor:
    """bf16 unit in the last place at |v| (float64; the smallest bf16 subnormal at 0)."""
    _, e = torch.frexp(v.abs())
    return torch.where(v == 0, torch.full_like(v, 2.0 ** -133), torch.ldexp(torch.ones_like(v), e - 8))


def gelu64(h: torch.Tensor) -> torch.Tensor:
    return 0.5 * h * (1.0 + torch.erf(h / math.sqrt(2.0)))


def gelu_grad64(h: torch.Tensor) -> torch.Tensor:
    return 0.5 * (1.0 + torch.erf(h / math.sqrt(2.0))) + h * torch.exp(-0.5 * h * h) / math.sqrt(2.0 * math.pi)


def product(a: torch.Tensor, b: torch.Tensor, bias: torch.Tensor | None = None):
    """(a b^T + bias, ACC (|a| |b|^T + |bias|)) in float64 for a [r, K], b [c, K]."""
    a, b = a.to(torch.float64), b.to(torch.float64)
    acc, bound = a @ b.T, a.abs() @ b.abs().T
    if bias is not None:
        bias = bias.to(torch.float64)
        acc += bias
        bound += bias.abs()
    return acc, ACC * bound


def contract_rows(a: torch.Tensor, b: torch.Tensor):
    """(a^T b, bound) in float64 for a [M, r], b [M, c]: the weight-gradient GEMMs, which contract over tokens (K = M, up to
    65 k). The bound is ACC |a|^T |b| plus RUN_SUM times the sum over the 64-token k-blocks of the running partial sum |S_kb|:
    every accumulation into the fp32 accumulator may be off by an fp32 ulp of the running sum, four of them per k-block. Where the
    partial sums grow steadily (dW2 = dh2^T h1 with h1 mostly positive holds db2 x mean(h1)) these errors add up linearly in K,
    which the first term, a random-walk size, does not cover."""
    acc = bound = run = None
    for r0 in range(0, a.shape[0], BLOCK_ROWS):
        ab = a[r0 : r0 + BLOCK_ROWS].to(torch.float64)
        bb = b[r0 : r0 + BLOCK_ROWS].to(torch.float64)
        q = ab.abs().T @ bb.abs()
        bound = q if bound is None else bound.add_(q)
        for s0 in range(0, ab.shape[0], KBLOCK):
            p = ab[s0 : s0 + KBLOCK].T @ bb[s0 : s0 + KBLOCK]
            acc = p if acc is None else acc.add_(p)
            run = acc.abs() if run is None else run.add_(acc.abs())
    return acc, ACC * bound + RUN_SUM * run


def gemm_error(epilogue: str, value: torch.Tensor, acc: torch.Tensor, bound: torch.Tensor, gelu_grad: torch.Tensor | None = None):
    """Per-element (|error|, tolerance) of a GEMM output ``value`` against the exact product ``acc`` (bias included) whose fp32
    accumulation error is at most ``bound``:
      "bf16"  (bias-GELU's h0, bias-sum-of-squares' h2): value = bf16(acc) -- half a bf16 ulp plus the accumulation bound;
      "dgelu" (dh0): value = bf16(bf16(acc) gelu'(h0)) -- one ulp at each rounding point, the accumulation bound through gelu',
              and the error of the epilogue's gelu';
      "f32"   (dW1, dW2): value = fp32(acc) -- the accumulation bound."""
    value = value.to(torch.float64)
    if epilogue == "bf16":
        return (value - acc).abs(), 0.5 * ulp(torch.maximum(value.abs(), acc.abs())) + bound
    if epilogue == "dgelu":
        t = bf16(acc)
        ref = bf16(t * gelu_grad)
        tol = (ulp(torch.maximum(value.abs(), ref.abs())) + gelu_grad.abs() * (ulp(torch.maximum(t.abs(), acc.abs())) + bound)
               + acc.abs() * GELU_GRAD_ABS)
        return (value - ref).abs(), tol
    if epilogue == "f32":
        return (value - acc).abs(), bound
    raise ValueError(epilogue)


def norm_mse(h2: torch.Tensor, g: torch.Tensor, target: torch.Tensor, eps: float, dy_coef: float) -> dict:
    """Rows of the fused norm + MSE + norm backward from the kernels' h2: rstd, y, diff = y - t, dy, dh2 (before its bf16
    rounding) and ``dh2_arith``, the size of the fp32 arithmetic that forms dh2 (|g| rstd (|y| + |diff|) dy_coef and the
    row-sum term): the kernel's dh2 is within one bf16 ulp plus ROW_EPS times that."""
    h = h2.to(torch.float64)
    gd = g.to(torch.float64)
    t = target.to(torch.float64)
    D = h.shape[1]
    rstd = torch.rsqrt(h.pow(2).mean(1, keepdim=True) + eps)
    xhat = h * rstd
    y = gd * xhat
    diff = y - t
    dy = dy_coef * diff
    s = (gd * dy * h).mean(1, keepdim=True)
    r3 = rstd.pow(3)
    dh2 = rstd * gd * dy - h * r3 * s
    row_terms = ((gd * h).abs() * (diff.abs() + y.abs())).sum(1, keepdim=True)
    dh2_arith = dy_coef * (gd.abs() * rstd * (y.abs() + diff.abs()) + h.abs() * r3 * row_terms / D) + (h * r3 * s).abs()
    return {"rstd": rstd.squeeze(1), "xhat": xhat, "y": y, "diff": diff, "dy": dy, "dh2": dh2, "dh2_arith": dh2_arith}
