"""The frozen T5 decoder's attention and feed-forward sublayers on packed rows (SURVEY section 8 f-1): host plumbing for the
relative position bias and the gated FFN's weight layout, and the autograd boundaries of their tcgen05 kernels. The attention
composes with ``frozen_linear`` for the Q / K / V / O projections."""
from __future__ import annotations

import math

import torch

from . import ops


def _decoder_bucket(n: torch.Tensor, num_buckets: int, max_distance: int) -> torch.Tensor:
    """transformers' ``T5Attention._relative_position_bucket(bidirectional=False)`` for distances ``n = i - j >= 0``: the first
    half of the buckets counts exact distances, the second half grows logarithmically up to ``max_distance`` (``log`` in fp32, then
    a truncating cast -- the exact arithmetic matters at the bucket edges)."""
    max_exact = num_buckets // 2
    large = max_exact + (torch.log(n.float() / max_exact) / math.log(max_distance / max_exact) * (num_buckets - max_exact)).to(torch.long)
    large = torch.minimum(large, torch.full_like(large, num_buckets - 1))
    return torch.where(n < max_exact, n, large)


def t5_position_bias_by_distance(table: torch.Tensor, num_buckets: int = 32, max_distance: int = 128) -> torch.Tensor:
    """Decoder self-attention bias as a per-distance table: ``table [num_buckets, H]`` (``relative_attention_bias.weight`` of block
    0) -> fp32 ``[H, max_distance]`` whose entry ``n`` is the bias of every (query i, key j = i - n) pair. Distances past the end
    use the last entry (the attention kernel clamps): for T5's bucket function every distance >= max_distance shares the bucket of
    ``max_distance - 1`` (the last one), so the clamped table equals ``T5Attention.compute_bias`` at any length."""
    if table.dim() != 2 or table.shape[0] != num_buckets:
        raise ValueError(f"table must be [num_buckets={num_buckets}, heads], got {tuple(table.shape)}")
    n = torch.arange(max_distance, device=table.device)
    bucket = _decoder_bucket(n, num_buckets, max_distance)
    if int(_decoder_bucket(torch.tensor([max_distance - 1]), num_buckets, max_distance)) != num_buckets - 1:
        raise ValueError("max_distance - 1 must fall in the last bucket for the clamped table to be exact")
    return table.detach()[bucket].t().float().contiguous()


class _T5Attention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, cu_q, cu_k, max_len_q, max_len_k, n_heads, bias):
        q, k, v = (t if t.dtype == torch.bfloat16 else t.to(torch.bfloat16) for t in (q, k, v))
        q, k, v = (t if t.stride(-1) == 1 and t.stride(0) % 8 == 0 else t.contiguous() for t in (q, k, v))
        need_lse = any(ctx.needs_input_grad[:3])
        o, lse = ops.t5_attention_fwd(q, k, v, cu_q, cu_k, max_len_q, max_len_k, n_heads, bias, need_lse=need_lse)
        if need_lse:
            ctx.save_for_backward(q, k, v, o, lse, cu_q, cu_k, bias)
        ctx.meta = (max_len_q, max_len_k, n_heads)
        return o

    @staticmethod
    def backward(ctx, do):
        q, k, v, o, lse, cu_q, cu_k, bias = ctx.saved_tensors
        max_len_q, max_len_k, n_heads = ctx.meta
        do = do.to(torch.bfloat16)
        if do.stride(-1) != 1 or do.stride(0) % 8:
            do = do.contiguous()
        dq, dk, dv = ops.t5_attention_bwd(do, q, k, v, o, lse, cu_q, cu_k, max_len_q, max_len_k, n_heads, bias)
        return dq, dk, dv, None, None, None, None, None, None


def t5_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, cu_q: torch.Tensor, cu_k: torch.Tensor | None, max_len_q: int,
                 max_len_k: int, n_heads: int, position_bias: torch.Tensor | None = None) -> torch.Tensor:
    """T5 attention core on packed rows, forward and backward on the library's tcgen05 kernels. Replaces the score / softmax / value
    product of transformers' ``T5Attention.forward`` (modeling_t5.py, ``scores = matmul(q, k^T)``, ``scores += position_bias``,
    ``softmax(scores.float())``, ``matmul(attn_weights, v)``) as called by the decoder of ``T5ForDecoder.forward``
    (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:211-224) -- without HF's padded batch, mask and bf16 scores:

    * cross-attention (``position_bias=None``): sample b's decoder rows ``q[cu_q[b]:cu_q[b+1]]`` attend to its packed aligner rows
      ``k / v[cu_k[b]:cu_k[b+1]]`` (K / V projected once on the packed rows, e.g. one ``frozen_linear`` with ``[Wk; Wv]``);
    * causal self-attention (``position_bias = t5_position_bias_by_distance(...)``): the rows attend to themselves, ``cu_k`` is
      None or ``cu_q``.

    ``q [Mq, 64 H]``, ``k / v [Mk, 64 H]`` (bf16; column slices of a fused projection output are read in place), ``cu_*`` int32
    device tensors, ``max_len_*`` host-known upper bounds of the samples' lengths. Returns ``[Mq, 64 H]`` bf16; the gradient flows to
    q, k and v (bf16), none to the frozen bias."""
    if position_bias is not None and position_bias.requires_grad:
        raise NotImplementedError("t5_attention: the position bias is frozen (no gradient); pass t5_position_bias_by_distance(...)")
    return _T5Attention.apply(q, k, v, cu_q, cu_k, int(max_len_q), int(max_len_k), int(n_heads), position_bias)


# ------------------------------------------------------------------------------------------------ feed-forward sublayer
_PAIR_ROWS = 32  # wi_0 / wi_1 interleave: one 32-column chunk of a GEMM epilogue warp (kEpiColsPerWarp / kEpiChunks)


def interleave_pairs(first: torch.Tensor, second: torch.Tensor, dim: int = 0) -> torch.Tensor:
    """The one place that knows the gated FFN's weight layout: ``first`` / ``second`` ([n, ...] along ``dim``, n % 32 == 0) ->
    ``[2 n, ...]`` whose blocks [64 k, 64 k + 32) are ``first[32 k : 32 k + 32]`` and [64 k + 32, 64 k + 64) ``second[32 k : 32 k +
    32]``. Applied to wi_0 / wi_1 (rows) it gives the ``wi`` the FFN kernels take; their ``ab`` / ``d_ab`` outputs come out in the same
    order along their columns. ``split_pairs`` inverts it. With 32 an epilogue warp's chunks 2j / 2j + 1 hold a matched (a, b) pair."""
    f, s = first.movedim(dim, 0), second.movedim(dim, 0)
    n = f.shape[0]
    if f.shape != s.shape or n % _PAIR_ROWS:
        raise ValueError(f"interleave_pairs: need two equal shapes with a multiple of {_PAIR_ROWS} along dim {dim}, got {tuple(first.shape)} and {tuple(second.shape)}")
    rest = tuple(f.shape[1:])
    out = torch.stack((f.reshape(n // _PAIR_ROWS, _PAIR_ROWS, *rest), s.reshape(n // _PAIR_ROWS, _PAIR_ROWS, *rest)), dim=1)
    return out.reshape(2 * n, *rest).movedim(0, dim).contiguous()


def split_pairs(t: torch.Tensor, dim: int = 0) -> tuple[torch.Tensor, torch.Tensor]:
    """Inverse of ``interleave_pairs``: ``[2 n, ...]`` along ``dim`` -> ``(first, second)``, e.g. ``ab`` -> ``(a, b)``."""
    u = t.movedim(dim, 0)
    n2 = u.shape[0]
    if n2 % (2 * _PAIR_ROWS):
        raise ValueError(f"split_pairs: size {n2} along dim {dim} is not a multiple of {2 * _PAIR_ROWS}")
    rest = tuple(u.shape[1:])
    v = u.reshape(n2 // (2 * _PAIR_ROWS), 2, _PAIR_ROWS, *rest)
    return tuple(v[:, i].reshape(n2 // 2, *rest).movedim(0, dim).contiguous() for i in (0, 1))


class T5FeedForwardWeights:
    """Frozen weights of one ``T5LayerFF`` (``T5DenseGatedActDense``, gated-gelu) in the layout the FFN kernels read: ``wi`` [2 d_ff,
    d] bf16 (wi_0 / wi_1 interleaved by ``interleave_pairs``), ``wo`` [d, d_ff] bf16, ``ln_weight`` [d] fp32 and ``eps``. Built once;
    ``split_pairs`` (also ``T5FeedForwardWeights.split``) undoes the interleave, e.g. on the ``ab`` / ``d_ab`` of ``ops.t5_ffn_*``."""

    split = staticmethod(split_pairs)

    def __init__(self, wi_0: torch.Tensor, wi_1: torch.Tensor, wo: torch.Tensor, ln_weight: torch.Tensor, eps: float = 1e-6):
        for t, n in ((wi_0, "wi_0"), (wi_1, "wi_1"), (wo, "wo"), (ln_weight, "layer_norm.weight")):
            if t.requires_grad:
                raise NotImplementedError(f"T5FeedForwardWeights: {n} must not require grad (the T5 decoder is frozen in ThinkDiff)")
        d_ff, d = wi_0.shape
        if tuple(wi_1.shape) != (d_ff, d) or tuple(wo.shape) != (d, d_ff) or tuple(ln_weight.shape) != (d,):
            raise ValueError(f"T5FeedForwardWeights: need wi_0 / wi_1 [d_ff, d], wo [d, d_ff], layer_norm.weight [d]; got "
                             f"{tuple(wi_0.shape)}, {tuple(wi_1.shape)}, {tuple(wo.shape)}, {tuple(ln_weight.shape)}")
        self.d, self.d_ff, self.eps = d, d_ff, float(eps)
        self.wi = interleave_pairs(wi_0.detach().to(torch.bfloat16), wi_1.detach().to(torch.bfloat16))
        self.wo = wo.detach().to(torch.bfloat16).contiguous()
        self.ln_weight = ln_weight.detach().float().contiguous()

    @classmethod
    def from_state_dict(cls, sd: dict, eps: float = 1e-6, prefix: str = "") -> "T5FeedForwardWeights":
        """From a ``T5LayerFF`` state dict (``layer_norm.weight``, ``DenseReluDense.wi_0/wi_1/wo.weight``, behind ``prefix``)."""
        return cls(sd[prefix + "DenseReluDense.wi_0.weight"], sd[prefix + "DenseReluDense.wi_1.weight"], sd[prefix + "DenseReluDense.wo.weight"],
                   sd[prefix + "layer_norm.weight"], eps)

    @classmethod
    def from_module(cls, layer) -> "T5FeedForwardWeights":
        """From a live transformers ``T5LayerFF`` whose parameters are frozen (``requires_grad_(False)``)."""
        ff = layer.DenseReluDense
        return cls(ff.wi_0.weight, ff.wi_1.weight, ff.wo.weight, layer.layer_norm.weight, layer.layer_norm.variance_epsilon)

    def to(self, device) -> "T5FeedForwardWeights":
        self.wi, self.wo, self.ln_weight = self.wi.to(device), self.wo.to(device), self.ln_weight.to(device)
        return self


class _T5LayerFF(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weights):
        x2 = x.reshape(-1, x.shape[-1]).to(torch.bfloat16).contiguous()
        need_grad = ctx.needs_input_grad[0]
        out, rstd, ab, _ = ops.t5_ffn_fwd(x2, weights.wi, weights.wo, weights.ln_weight, weights.eps, want_ab=need_grad)
        if need_grad:
            ctx.save_for_backward(x2, rstd, ab)
            ctx.weights = weights
        ctx.shape, ctx.dtype = x.shape, x.dtype
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, rstd, ab = ctx.saved_tensors
        w = ctx.weights
        dy2 = dy.reshape(x2.shape).to(torch.bfloat16).contiguous()
        dx, _ = ops.t5_ffn_bwd(dy2, x2, rstd, ab, w.wi, w.wo, w.ln_weight)
        return dx.view(ctx.shape).to(ctx.dtype), None


def t5_layer_ff(x: torch.Tensor, weights: T5FeedForwardWeights) -> torch.Tensor:
    """transformers' ``T5LayerFF`` with ``T5DenseGatedActDense`` (Flan-T5's gated-gelu FFN) on packed decoder rows, forward and input
    gradient on the library's kernels: ``x + wo(gelu_new(wi_0(norm(x))) * wi_1(norm(x)))`` with the rounding of the bf16 model under
    bf16 autocast, dropout off (DESIGN.md section 7). ``x [..., d]``; returns bf16 of the same shape. The weights are frozen: the
    gradient flows to ``x`` only. Saves ``x``, ``rstd`` and ``ab`` ([rows, 2 d_ff] bf16) for the backward."""
    return _T5LayerFF.apply(x, weights)
