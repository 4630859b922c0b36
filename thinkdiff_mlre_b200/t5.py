"""The frozen T5 decoder's attention on packed rows (SURVEY section 8 f-1): host plumbing for the relative position bias and the
autograd boundary of the tcgen05 attention kernels. Composes with ``frozen_linear`` for the Q / K / V / O projections."""
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
