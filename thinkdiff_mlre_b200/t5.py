"""The frozen T5 decoder on packed rows (SURVEY section 8 f-1): host plumbing for the relative position bias and the gated FFN's
weight layout, the autograd boundaries of the attention core and of the three sublayers (self-attention, cross-attention,
feed-forward), and their composition into a decoder block and the decoder stack. The attention core also composes with
``frozen_linear`` for hand-built projections."""
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


# ------------------------------------------------------------------------------------------------ attention sublayers, block, stack
def _frozen(named):
    for n, t in named:
        if t.requires_grad:
            raise NotImplementedError(f"T5 decoder weights: {n} must not require grad (the T5 decoder is frozen in ThinkDiff)")


class T5DecoderBlockWeights:
    """Frozen weights of one decoder ``T5Block`` in the layout the sublayer kernels read: the three pre-norm weights ``ln_self``,
    ``ln_cross`` (fp32 [d]) and ``ffn.ln_weight``; ``w_qkv`` [3 inner, d] (``[Wq; Wk; Wv]`` of the self-attention, one GEMM),
    ``wo_self`` [d, inner], ``w_q`` [inner, d], ``w_kv`` [2 inner, d] (``[Wk; Wv]`` of the cross-attention) and ``wo_cross`` [d, inner]
    (bf16); ``ffn`` (``T5FeedForwardWeights``); ``n_heads`` and ``eps``. inner = 64 n_heads: d_kv must be 64."""

    def __init__(self, ln_self, wq, wk, wv, wo_self, ln_cross, cq, ck, cv, wo_cross, ffn: T5FeedForwardWeights, n_heads: int,
                 eps: float = 1e-6):
        _frozen((("layer.0.layer_norm.weight", ln_self), ("SelfAttention.q", wq), ("SelfAttention.k", wk), ("SelfAttention.v", wv),
                 ("SelfAttention.o", wo_self), ("layer.1.layer_norm.weight", ln_cross), ("EncDecAttention.q", cq),
                 ("EncDecAttention.k", ck), ("EncDecAttention.v", cv), ("EncDecAttention.o", wo_cross)))
        inner, d = wq.shape
        if n_heads < 1 or inner != 64 * n_heads:
            raise NotImplementedError(f"T5DecoderBlockWeights: d_kv = {inner / max(n_heads, 1):g} (inner {inner}, {n_heads} heads); the "
                                      "attention kernels need d_kv = 64")
        for t, shape, n in ((wk, (inner, d), "k"), (wv, (inner, d), "v"), (cq, (inner, d), "cross q"), (ck, (inner, d), "cross k"),
                            (cv, (inner, d), "cross v"), (wo_self, (d, inner), "o"), (wo_cross, (d, inner), "cross o"),
                            (ln_self, (d,), "layer.0.layer_norm"), (ln_cross, (d,), "layer.1.layer_norm")):
            if tuple(t.shape) != shape:
                raise ValueError(f"T5DecoderBlockWeights: {n} must be {list(shape)}, got {list(t.shape)}")
        if ffn.d != d:
            raise ValueError(f"T5DecoderBlockWeights: the FFN's d = {ffn.d} differs from the attention's d = {d}")

        def bf(*ts):
            return torch.cat([t.detach().to(torch.bfloat16) for t in ts]).contiguous()

        self.d, self.n_heads, self.eps = d, int(n_heads), float(eps)
        self.ln_self, self.ln_cross = ln_self.detach().float().contiguous(), ln_cross.detach().float().contiguous()
        self.w_qkv, self.wo_self = bf(wq, wk, wv), bf(wo_self)
        self.w_q, self.w_kv, self.wo_cross = bf(cq), bf(ck, cv), bf(wo_cross)
        self.ffn = ffn

    @classmethod
    def from_module(cls, block) -> "T5DecoderBlockWeights":
        """From a live transformers decoder ``T5Block`` whose parameters are frozen (``requires_grad_(False)``)."""
        sa, ca = block.layer[0], block.layer[1]
        a, c = sa.SelfAttention, ca.EncDecAttention
        if a.key_value_proj_dim != 64 or c.key_value_proj_dim != 64:
            raise NotImplementedError(f"T5DecoderBlockWeights: d_kv = {a.key_value_proj_dim}; the attention kernels need d_kv = 64")
        return cls(sa.layer_norm.weight, a.q.weight, a.k.weight, a.v.weight, a.o.weight, ca.layer_norm.weight, c.q.weight, c.k.weight,
                   c.v.weight, c.o.weight, T5FeedForwardWeights.from_module(block.layer[2]), a.n_heads, sa.layer_norm.variance_epsilon)

    @classmethod
    def from_state_dict(cls, sd: dict, n_heads: int, eps: float = 1e-6, prefix: str = "") -> "T5DecoderBlockWeights":
        """From a ``T5Block`` state dict (``layer.0.SelfAttention.q.weight``, ..., behind ``prefix``, e.g. ``"block.3."``)."""
        s, c = prefix + "layer.0.", prefix + "layer.1."
        return cls(sd[s + "layer_norm.weight"], *(sd[s + f"SelfAttention.{n}.weight"] for n in "qkvo"), sd[c + "layer_norm.weight"],
                   *(sd[c + f"EncDecAttention.{n}.weight"] for n in "qkvo"),
                   T5FeedForwardWeights.from_state_dict(sd, eps, prefix=prefix + "layer.2."), n_heads, eps)

    def to(self, device) -> "T5DecoderBlockWeights":
        for n in ("ln_self", "ln_cross", "w_qkv", "wo_self", "w_q", "w_kv", "wo_cross"):
            setattr(self, n, getattr(self, n).to(device))
        self.ffn.to(device)
        return self


class T5DecoderWeights:
    """Frozen weights of a decoder ``T5Stack``: ``blocks`` (``T5DecoderBlockWeights``), ``final_ln`` (fp32 [d]), ``eps``, and
    ``position_bias``, block 0's relative attention bias table turned once into the per-distance table the self-attention kernels
    read (``t5_position_bias_by_distance``, [H, max_distance] fp32), shared by every block as in HF."""

    def __init__(self, blocks, final_ln: torch.Tensor, bias_table: torch.Tensor, eps: float = 1e-6, num_buckets: int = 32,
                 max_distance: int = 128):
        _frozen((("final_layer_norm.weight", final_ln), ("relative_attention_bias.weight", bias_table)))
        self.blocks = list(blocks)
        if not self.blocks:
            raise ValueError("T5DecoderWeights: no blocks")
        self.final_ln = final_ln.detach().float().contiguous()
        self.position_bias = t5_position_bias_by_distance(bias_table, num_buckets, max_distance)
        if self.position_bias.shape[0] != self.blocks[0].n_heads:
            raise ValueError(f"T5DecoderWeights: the bias table has {self.position_bias.shape[0]} heads, the blocks {self.blocks[0].n_heads}")
        self.eps = float(eps)

    @classmethod
    def from_module(cls, stack) -> "T5DecoderWeights":
        """From a live transformers decoder ``T5Stack`` whose parameters are frozen."""
        cfg = stack.config
        return cls([T5DecoderBlockWeights.from_module(b) for b in stack.block], stack.final_layer_norm.weight,
                   stack.block[0].layer[0].SelfAttention.relative_attention_bias.weight, stack.final_layer_norm.variance_epsilon,
                   cfg.relative_attention_num_buckets, cfg.relative_attention_max_distance)

    @classmethod
    def from_state_dict(cls, sd: dict, n_heads: int, eps: float = 1e-6, prefix: str = "", num_buckets: int = 32,
                        max_distance: int = 128) -> "T5DecoderWeights":
        """From a decoder ``T5Stack`` state dict (``block.{i}.layer...``, ``final_layer_norm.weight``, behind ``prefix``)."""
        n_blocks = 1 + max(int(k[len(prefix):].split(".")[1]) for k in sd if k.startswith(prefix + "block."))
        blocks = [T5DecoderBlockWeights.from_state_dict(sd, n_heads, eps, prefix=f"{prefix}block.{i}.") for i in range(n_blocks)]
        return cls(blocks, sd[prefix + "final_layer_norm.weight"], sd[prefix + "block.0.layer.0.SelfAttention.relative_attention_bias.weight"],
                   eps, num_buckets, max_distance)

    def to(self, device) -> "T5DecoderWeights":
        for b in self.blocks:
            b.to(device)
        self.final_ln, self.position_bias = self.final_ln.to(device), self.position_bias.to(device)
        return self


class _T5LayerSelfAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, cu_q, max_len, weights, bias):
        w = weights
        x2 = x.reshape(-1, x.shape[-1]).to(torch.bfloat16).contiguous()
        need_grad = ctx.needs_input_grad[0]
        out, rstd, qkv, o, lse = ops.t5_self_attention_layer_fwd(x2, w.w_qkv, w.wo_self, w.ln_self, w.eps, bias, cu_q, max_len, w.n_heads,
                                                                 want_saved=need_grad)
        if need_grad:
            ctx.save_for_backward(x2, rstd, qkv, o, lse, cu_q, bias)
            ctx.weights, ctx.max_len = w, max_len
        ctx.shape, ctx.dtype = x.shape, x.dtype
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, rstd, qkv, o, lse, cu_q, bias = ctx.saved_tensors
        w = ctx.weights
        dy2 = dy.reshape(x2.shape).to(torch.bfloat16).contiguous()
        dx, _ = ops.t5_self_attention_layer_bwd(dy2, x2, rstd, qkv, o, lse, w.w_qkv, w.wo_self, w.ln_self, bias, cu_q, ctx.max_len, w.n_heads)
        return dx.view(ctx.shape).to(ctx.dtype), None, None, None, None


def t5_layer_self_attention(x: torch.Tensor, cu_q: torch.Tensor, max_len_q: int, weights: T5DecoderBlockWeights,
                            position_bias: torch.Tensor) -> torch.Tensor:
    """transformers' ``T5LayerSelfAttention`` of a decoder block on packed rows, forward and input gradient on the library's kernels:
    ``x + o(attention(q(norm(x)), k(norm(x)), v(norm(x))))``, causal within each sample ``cu_q[b]:cu_q[b+1]`` (covering every row),
    with ``position_bias`` from ``T5DecoderWeights.position_bias`` (or ``t5_position_bias_by_distance``), rounded as the bf16 model
    under bf16 autocast (DESIGN.md section 7). ``x [rows, d]``; returns bf16. The weights are frozen: the gradient flows to ``x``.
    Saves ``x``, ``rstd``, ``qkv``, ``o`` and ``lse`` when ``x`` needs a gradient, nothing otherwise."""
    if position_bias is None or position_bias.requires_grad:
        raise NotImplementedError("t5_layer_self_attention: pass the frozen per-distance bias table (t5_position_bias_by_distance)")
    return _T5LayerSelfAttention.apply(x, cu_q, int(max_len_q), weights, position_bias)


class _T5LayerCrossAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, enc, cu_q, cu_k, max_len_q, max_len_k, weights):
        w = weights
        x2 = x.reshape(-1, x.shape[-1]).to(torch.bfloat16).contiguous()
        e2 = enc.reshape(-1, enc.shape[-1]).to(torch.bfloat16).contiguous()  # autocast's cast, once per use as in HF
        need_grad = any(ctx.needs_input_grad[:2])
        out, rstd, q, kv, o, lse = ops.t5_cross_attention_layer_fwd(x2, e2, w.w_q, w.w_kv, w.wo_cross, w.ln_cross, w.eps, cu_q, cu_k,
                                                                    max_len_q, max_len_k, w.n_heads, want_saved=need_grad)
        if need_grad:
            ctx.save_for_backward(x2, rstd, q, kv, o, lse, cu_q, cu_k)
            ctx.weights, ctx.max_lens = w, (max_len_q, max_len_k)
        ctx.shapes, ctx.dtypes = (x.shape, enc.shape), (x.dtype, enc.dtype)
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, rstd, q, kv, o, lse, cu_q, cu_k = ctx.saved_tensors
        w = ctx.weights
        dy2 = dy.reshape(x2.shape).to(torch.bfloat16).contiguous()
        dx, d_enc = ops.t5_cross_attention_layer_bwd(dy2, x2, rstd, q, kv, o, lse, w.w_q, w.w_kv, w.wo_cross, w.ln_cross, cu_q, cu_k,
                                                     *ctx.max_lens, w.n_heads)
        # d_enc is fp32: returned in enc's dtype, so autograd sums the blocks' contributions in fp32 when enc is fp32
        d_enc = d_enc.view(ctx.shapes[1]).to(ctx.dtypes[1]) if ctx.needs_input_grad[1] else None
        dx = dx.view(ctx.shapes[0]).to(ctx.dtypes[0]) if ctx.needs_input_grad[0] else None
        return dx, d_enc, None, None, None, None, None


def t5_layer_cross_attention(x: torch.Tensor, enc: torch.Tensor, cu_q: torch.Tensor, cu_k: torch.Tensor, max_len_q: int, max_len_k: int,
                             weights: T5DecoderBlockWeights) -> torch.Tensor:
    """transformers' ``T5LayerCrossAttention`` on packed rows: decoder rows ``x`` (samples ``cu_q``) attend to the packed aligner rows
    ``enc [Mk, d]`` (samples ``cu_k``), ``x + o(attention(q(norm(x)), k(enc), v(enc)))``. ``enc`` may be fp32 (the aligner's output in
    training) or bf16; it is cast to bf16 inside, and its gradient, summed in fp32 by one GEMM, comes back in ``enc``'s dtype. A sample
    without aligner rows passes ``x`` through unchanged. Returns bf16 of ``x``'s shape."""
    return _T5LayerCrossAttention.apply(x, enc, cu_q, cu_k, int(max_len_q), int(max_len_k), weights)


def t5_decoder_block(x: torch.Tensor, enc: torch.Tensor, cu_q: torch.Tensor, cu_k: torch.Tensor, max_len_q: int, max_len_k: int,
                     weights: T5DecoderBlockWeights, position_bias: torch.Tensor) -> torch.Tensor:
    """One decoder ``T5Block`` on packed rows: causal self-attention with the relative position bias, cross-attention to the packed
    aligner rows, gated-GELU FFN, each pre-norm with its residual, on the library's kernels (15 launches forward, 19 backward)."""
    h = t5_layer_self_attention(x, cu_q, max_len_q, weights, position_bias)
    h = t5_layer_cross_attention(h, enc, cu_q, cu_k, max_len_q, max_len_k, weights)
    return t5_layer_ff(h, weights.ffn)


class _T5FinalNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, eps):
        x2 = x.reshape(-1, x.shape[-1]).to(torch.bfloat16).contiguous()
        y, rstd = ops.rmsnorm_fwd(x2, weight, eps, out_bf16=True)
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(x2, rstd, weight)
        ctx.shape, ctx.dtype = x.shape, x.dtype
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, rstd, weight = ctx.saved_tensors
        dy2 = dy.reshape(x2.shape).to(torch.bfloat16).contiguous()
        dx, _, _ = ops.rmsnorm_bwd(dy2, x2, rstd, weight, want_dg=False, want_dxsum=False)
        return dx.view(ctx.shape).to(ctx.dtype), None, None


def t5_decoder_stack(dec_rows: torch.Tensor, enc: torch.Tensor, cu_q: torch.Tensor, cu_k: torch.Tensor, max_len_q: int, max_len_k: int,
                     weights: T5DecoderWeights) -> torch.Tensor:
    """The frozen decoder ``T5Stack`` of ``T5ForDecoder.forward`` (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:211-224) on packed
    rows: every block in order (``t5_decoder_block``), then the frozen final norm (bf16 out; its backward skips the weight gradient).
    ``dec_rows [Mq, d]`` are the decoder input embeddings packed with ``cu_q``; ``enc [Mk, d]`` the aligner rows packed with ``cu_k``
    (fp32 or bf16; the gradient reaching it is summed over the blocks in its dtype). With right-padded labels and no decoder mask, as
    in the reference, a valid position never sees a pad position under the causal mask, so packing only the valid decoder rows is exact
    for the loss. The output feeds ``lm_head_cross_entropy`` unchanged."""
    h = dec_rows
    for bw in weights.blocks:
        h = t5_decoder_block(h, enc, cu_q, cu_k, max_len_q, max_len_k, bw, weights.position_bias)
    return _T5FinalNorm.apply(h, weights.final_ln, weights.eps)


# ------------------------------------------------------------------------------------------------ the objective: labels -> CE -> enc grad
IGNORE_INDEX = -100


def pack_labels(labels: torch.Tensor, vocab_size: int):
    """The tokenizer's right-padded labels ``[B, T]`` int64 (-100 = ignored) -> ``(flat int64 [Mq], lens int32 [B], max_len_q)`` on
    ``labels``' device: sample b keeps its positions up to and including its last label that is not -100 (none when all are -100),
    interior -100s included -- the loss ignores them and the decoder input after them is the pad token, as in HF. Packing is exact for
    the loss: under the causal mask a kept position never sees a dropped one, and dropped positions carry no loss. Rejects labels
    outside [0, vocab_size) other than -100 (the decoder-input kernel would give them a zero row, HF an index error)."""
    if labels.dim() != 2 or labels.dtype != torch.int64:
        raise TypeError(f"pack_labels: labels must be int64 [B, T], got {labels.dtype} {tuple(labels.shape)}")
    keep = labels != IGNORE_INDEX
    bad = keep & ((labels < 0) | (labels >= vocab_size))
    if bool(bad.any()):
        raise ValueError(f"pack_labels: label ids must be -100 or in [0, {vocab_size}); got {labels[bad][:4].tolist()}")
    pos = torch.arange(1, labels.shape[1] + 1, device=labels.device)
    lens = (keep * pos).amax(dim=1) if labels.shape[1] else torch.zeros(labels.shape[0], dtype=torch.int64, device=labels.device)
    flat = labels[pos[None, :] <= lens[:, None]]
    return flat.contiguous(), lens.to(torch.int32), int(lens.max()) if lens.numel() else 0


def _scales_decoder_output(cfg) -> bool:
    """Whether the model multiplies the decoder output by d_model^-0.5 before ``lm_head``: ``scale_decoder_outputs`` in transformers
    5.x, ``tie_word_embeddings`` before it (4.46.1: ``if self.config.tie_word_embeddings: sequence_output *= model_dim**-0.5``)."""
    scale = getattr(cfg, "scale_decoder_outputs", None)
    return bool(getattr(cfg, "tie_word_embeddings", True) if scale is None else scale)


class T5ForDecoderWeights:
    """Frozen weights of the reference's objective (``T5ForDecoder.forward``, thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:211-246):
    ``decoder`` (``T5DecoderWeights``), ``embed`` and ``lm_head`` ([V, d] bf16), ``decoder_start_token_id`` and ``pad_token_id``. Only the
    unscaled head is built (Flan-T5-XXL's, untied in its config): a configuration that scales the decoder output before ``lm_head`` is
    rejected."""

    def __init__(self, decoder: T5DecoderWeights, embed: torch.Tensor, lm_head: torch.Tensor, decoder_start_token_id: int = 0,
                 pad_token_id: int = 0):
        _frozen((("embed_tokens.weight", embed), ("lm_head.weight", lm_head)))
        d = decoder.blocks[0].d
        if embed.dim() != 2 or embed.shape[1] != d or tuple(lm_head.shape) != tuple(embed.shape):
            raise ValueError(f"T5ForDecoderWeights: need embed and lm_head [V, {d}], got {tuple(embed.shape)} and {tuple(lm_head.shape)}")
        if d % 8:
            raise ValueError(f"T5ForDecoderWeights: d = {d} must be a multiple of 8")
        self.decoder = decoder
        self.embed = embed.detach().to(torch.bfloat16).contiguous()
        self.lm_head = lm_head.detach().to(torch.bfloat16).contiguous()
        self.vocab_size = int(embed.shape[0])
        self.decoder_start_token_id, self.pad_token_id = int(decoder_start_token_id), int(pad_token_id)
        for n, t in (("decoder_start_token_id", self.decoder_start_token_id), ("pad_token_id", self.pad_token_id)):
            if not 0 <= t < self.vocab_size:
                raise ValueError(f"T5ForDecoderWeights: {n} = {t} is outside [0, {self.vocab_size})")

    @staticmethod
    def _check_config(cfg):
        if _scales_decoder_output(cfg):
            raise NotImplementedError("T5ForDecoderWeights: this configuration scales the decoder output by d_model^-0.5 before lm_head "
                                      "(tie_word_embeddings / scale_decoder_outputs); only the unscaled head (Flan-T5) is built")

    @classmethod
    def from_module(cls, model) -> "T5ForDecoderWeights":
        """From a live transformers ``T5ForConditionalGeneration`` whose decoder, embedding and head are frozen."""
        cfg = model.config
        cls._check_config(cfg)
        return cls(T5DecoderWeights.from_module(model.decoder), model.get_input_embeddings().weight, model.lm_head.weight,
                   cfg.decoder_start_token_id, cfg.pad_token_id)

    @classmethod
    def from_state_dict(cls, sd: dict, config) -> "T5ForDecoderWeights":
        """From a ``T5ForConditionalGeneration`` state dict (``decoder.block.{i}...``, ``decoder.final_layer_norm.weight``,
        ``shared.weight``, ``lm_head.weight``) and its ``T5Config``."""
        cls._check_config(config)
        dec = T5DecoderWeights.from_state_dict(sd, config.num_heads, config.layer_norm_epsilon, prefix="decoder.",
                                               num_buckets=config.relative_attention_num_buckets,
                                               max_distance=config.relative_attention_max_distance)
        embed = sd["shared.weight"] if "shared.weight" in sd else sd["decoder.embed_tokens.weight"]
        return cls(dec, embed, sd["lm_head.weight"], config.decoder_start_token_id, config.pad_token_id)

    def to(self, device) -> "T5ForDecoderWeights":
        self.decoder.to(device)
        self.embed, self.lm_head = self.embed.to(device), self.lm_head.to(device)
        return self


class _T5DecoderLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc, cu_k, max_len_k, labels, cu_q, max_len_q, weights):
        e2 = enc.reshape(-1, enc.shape[-1])
        loss, d_enc = ops.t5_decoder_loss_fwd_bwd(e2, cu_k, max_len_k, labels, cu_q, max_len_q, weights, 1.0, want_grad=True)
        ctx.d_enc, ctx.shape, ctx.dtype = d_enc, enc.shape, enc.dtype
        return loss

    @staticmethod
    def backward(ctx, g):
        d_enc = ctx.d_enc
        ctx.d_enc = None
        return d_enc.mul_(g.to(d_enc.dtype)).view(ctx.shape).to(ctx.dtype), None, None, None, None, None, None


def t5_decoder_loss(enc: torch.Tensor, cu_k: torch.Tensor, max_len_k: int, labels: torch.Tensor, cu_q: torch.Tensor, max_len_q: int,
                    weights: T5ForDecoderWeights) -> torch.Tensor:
    """The loss of ``T5ForDecoder.forward(encoder_outputs=..., labels=...)`` (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:211-246,
    called at :590-598) on packed rows: ``CrossEntropyLoss(ignore_index=-100)`` of the frozen decoder's logits, the decoder reading its
    inputs from the labels (``_shift_right`` + ``embed_tokens``) and cross-attending to the aligner rows. ``enc [Mk, d]`` (fp32 in
    training, or bf16) packed with ``cu_k``; ``labels`` / ``cu_q`` / ``max_len_q`` from ``pack_labels`` (``cu_q = ops.cu_seqlens(lens)``).

    One autograd node over ``ops.t5_decoder_loss_fwd_bwd``: the gradient is formed in the forward, summed over the blocks in fp32, and
    the backward multiplies it by the upstream scalar; it reaches ``enc`` in ``enc``'s dtype, never rounded to bf16 on the way. Without
    a gradient to form (``no_grad``, or ``enc`` not requiring one) only the forward runs and nothing is kept."""
    if torch.is_grad_enabled() and enc.requires_grad:
        return _T5DecoderLoss.apply(enc, cu_k, int(max_len_k), labels, cu_q, int(max_len_q), weights)
    loss, _ = ops.t5_decoder_loss_fwd_bwd(enc.detach().reshape(-1, enc.shape[-1]), cu_k, int(max_len_k), labels, cu_q, int(max_len_q), weights,
                                          want_grad=False)
    return loss
