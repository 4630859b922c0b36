"""fp32 reference of the T5 attention kernels (csrc/attn_sm100.cuh) on PACKED rows -- test infrastructure only, the product path
never imports it. tests/test_t5_attention_cpu.py pins it live to transformers' ``T5Attention`` on the zero-padded batch + mask;
tests/test_gpu_t5_attention.py compares the kernels against it."""
from __future__ import annotations

import torch


def attention_packed(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, cu_q, cu_k, n_heads: int, bias_by_distance: torch.Tensor | None = None,
                     return_lse: bool = False):
    """The attention core of both decoder sublayers on PACKED rows, in fp32: sample ``b``'s queries ``q[cu_q[b]:cu_q[b+1]]`` attend to
    keys / values ``k / v[cu_k[b]:cu_k[b+1]]`` (``[rows, H * dk]``, head h = columns h*dk..). ``bias_by_distance [H, n_dist]`` given:
    causal self-attention (keys = the query rows, ``cu_k`` ignored) with bias entry ``min(i - j, n_dist - 1)`` for query position
    i >= key position j, positions counted from the sample's first row. No scaling (T5). A sample without keys gets zeros (and
    lse = -inf). ``return_lse``: also the natural-log normaliser ``[H, Mq]``."""
    q, k, v = q.float(), k.float(), v.float()
    cu_q = [int(c) for c in cu_q]
    cu_k = cu_q if bias_by_distance is not None else [int(c) for c in cu_k]
    dk = q.shape[1] // n_heads

    def heads(x):  # [L, H*dk] -> [H, L, dk], also for empty samples
        return x.reshape(x.shape[0], n_heads, dk).transpose(0, 1)

    outs, lses = [], []
    for b in range(len(cu_q) - 1):
        qh = heads(q[cu_q[b] : cu_q[b + 1]])
        kh, vh = heads(k[cu_k[b] : cu_k[b + 1]]), heads(v[cu_k[b] : cu_k[b + 1]])
        s = qh @ kh.transpose(-1, -2)  # [H, T, L]
        if bias_by_distance is not None:
            T = s.shape[1]
            n = torch.arange(T)[:, None] - torch.arange(T)[None, :]
            bias = bias_by_distance.float()[:, n.clamp(0, bias_by_distance.shape[1] - 1)]
            s = (s + bias).masked_fill(n < 0, float("-inf"))
        lse = torch.logsumexp(s, dim=-1)  # [H, T]
        p = torch.exp(s - lse[..., None]) if s.shape[-1] > 0 else s
        outs.append((p @ vh).transpose(0, 1).reshape(qh.shape[1], n_heads * dk))
        lses.append(lse)
    o = torch.cat(outs) if outs else q.new_zeros((0, q.shape[1]))
    if return_lse:
        return o, (torch.cat(lses, dim=1) if lses else q.new_zeros((n_heads, 0)))
    return o
