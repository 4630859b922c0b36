"""Functional wrappers: torch tensors in, C-ABI calls out. torch is used for device memory and streams only.

Every function checks shapes/dtypes on the host, allocates outputs through the caching allocator (so stream
semantics hold) and launches on ``torch.cuda.current_stream()``.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("thinkdiff_mlre_b200 runs on CUDA tensors only (no CPU fallback)")


def _contig(t, name):
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


# ------------------------------------------------------------------------------------------------ pack
def cu_seqlens(lens: torch.Tensor) -> torch.Tensor:
    """int32 lens[B] (device) -> int32 cu_seqlens[B+1] (device)."""
    _need_cuda(lens)
    lens = _contig(lens.to(torch.int32), "lens")
    cu = torch.empty(lens.numel() + 1, dtype=torch.int32, device=lens.device)
    L.launch_count += 1
    L.check(L.lib().td_cu_seqlens(L.ptr(lens), lens.numel(), L.ptr(cu), L.stream_ptr()), "td_cu_seqlens")
    return cu


def pack_varlen(flat: torch.Tensor, src_row_start: torch.Tensor, cu: torch.Tensor, total_rows: int, want_index: bool = False):
    """flat [R, C] (any dtype) -> packed [total_rows, C]: rows src_row_start[i] + [0, len_i) of each sample, back to back.
    ``want_index``: also return int64 [total_rows] = the source row of every packed row."""
    _need_cuda(flat, src_row_start, cu)
    _contig(flat, "flat")
    if src_row_start.dtype != torch.int64 or cu.dtype != torch.int32:
        raise TypeError("src_row_start must be int64 and cu_seqlens int32")
    out = torch.empty((total_rows, flat.shape[1]), dtype=flat.dtype, device=flat.device)
    index = torch.empty((total_rows,), dtype=torch.int64, device=flat.device) if want_index else None
    row_bytes = flat.shape[1] * flat.element_size()
    L.launch_count += 1
    L.check(
        L.lib().td_pack_varlen_indexed(L.ptr(flat), L.ptr(src_row_start), L.ptr(cu), cu.numel() - 1, total_rows, row_bytes,
                                       L.ptr(out), L.ptr(index), L.stream_ptr()),
        "td_pack_varlen",
    )
    return (out, index) if want_index else out


def pack_varlen2(src: torch.Tensor, src2: torch.Tensor, src_row_start: torch.Tensor, cu: torch.Tensor, total_rows: int):
    """Gather ragged segments of TWO tensors ``[R1, C]`` / ``[R2, C]`` into one packed ``[total_rows, C]`` with a single launch:
    segment i reads rows ``src_row_start[i]..`` of ``src`` when that is >= 0, rows ``-(src_row_start[i] + 1)..`` of ``src2`` otherwise."""
    _need_cuda(src, src2, src_row_start, cu)
    _contig(src, "src")
    _contig(src2, "src2")
    if src.shape[1:] != src2.shape[1:] or src.dtype != src2.dtype:
        raise ValueError("pack_varlen2: the two sources must agree in row shape and dtype")
    if src_row_start.dtype != torch.int64 or cu.dtype != torch.int32:
        raise TypeError("src_row_start must be int64 and cu_seqlens int32")
    out = torch.empty((total_rows, src.shape[1]), dtype=src.dtype, device=src.device)
    row_bytes = src.shape[1] * src.element_size()
    L.launch_count += 1
    L.check(L.lib().td_pack_varlen2(L.ptr(src), L.ptr(src2), L.ptr(src_row_start), L.ptr(cu), cu.numel() - 1, total_rows, row_bytes,
                                    L.ptr(out), L.stream_ptr()), "td_pack_varlen2")
    return out


def pack_padded(flat: torch.Tensor, src_row_start: torch.Tensor, cu: torch.Tensor, l_max: int, want_mask: bool = True):
    """Reference layout: zero-padded [B, l_max, C] and int64 mask [B, l_max]."""
    _need_cuda(flat, src_row_start, cu)
    _contig(flat, "flat")
    B = cu.numel() - 1
    out = torch.empty((B, l_max, flat.shape[1]), dtype=flat.dtype, device=flat.device)
    mask = torch.empty((B, l_max), dtype=torch.int64, device=flat.device) if want_mask else None
    row_bytes = flat.shape[1] * flat.element_size()
    L.launch_count += 1
    L.check(
        L.lib().td_pack_padded(L.ptr(flat), L.ptr(src_row_start), L.ptr(cu), B, l_max, row_bytes, L.ptr(out), L.ptr(mask),
                               L.stream_ptr()),
        "td_pack_padded",
    )
    return out, mask


# ------------------------------------------------------------------------------------------------ params
def cast_to_bf16(src: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    _need_cuda(src)
    if src.dtype != torch.float32:
        raise TypeError("cast_to_bf16 expects float32")
    _contig(src, "src")
    if out is None:
        out = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    L.launch_count += 1
    L.check(L.lib().td_cast_f32_to_bf16(L.ptr(src), L.ptr(out), src.numel(), L.stream_ptr()), "td_cast_f32_to_bf16")
    return out


# ------------------------------------------------------------------------------------------------ aligner
def aligner_fwd(x, W1, b1, W2, b2, g, eps: float, out_bf16: bool, save_for_backward: bool):
    """x [M, Din] bf16; W/b bf16; g fp32 -> y [M, D] (fp32, or bf16 when out_bf16), saved = (h0, h1, h2, rstd)."""
    _need_cuda(x, W1, W2, g)
    M, Din = x.shape
    D = W1.shape[0]
    for t, n in ((x, "x"), (W1, "W1"), (W2, "W2")):
        if t.dtype != torch.bfloat16:
            raise TypeError(f"{n} must be bfloat16")
        _contig(t, n)
    if g.dtype != torch.float32:
        raise TypeError("norm weight must be float32 at the ABI")
    dev = x.device
    h0 = torch.empty((M, D), dtype=torch.bfloat16, device=dev) if save_for_backward else None
    h1 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
    h2 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
    rstd = torch.empty((M,), dtype=torch.float32, device=dev)
    y = torch.empty((M, D), dtype=torch.bfloat16 if out_bf16 else torch.float32, device=dev)
    ws_bytes = L.lib().td_aligner_fwd_workspace_bytes(M, Din, D)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.launch_count += 3
    L.check(
        L.lib().td_aligner_fwd(L.ptr(x), M, Din, D, L.ptr(W1), L.ptr(b1), L.ptr(W2), L.ptr(b2), L.ptr(g), eps, L.ptr(h0),
                               L.ptr(h1), L.ptr(h2), L.ptr(rstd), L.ptr(y), L.BF16 if out_bf16 else L.F32, L.ptr(ws),
                               ws_bytes, L.stream_ptr()),
        "td_aligner_fwd",
    )
    return y, (h0, h1, h2, rstd)


class AlignerBackward:
    """Two-phase aligner backward writing into caller-chosen gradient buffers (so buckets can be flat)."""

    def __init__(self, x, saved, W2, g, dy, grad_scale: float = 1.0):
        self.x, (self.h0, self.h1, self.h2, self.rstd), self.W2, self.g = x, saved, W2, g
        self.dy = _contig(dy, "dy")
        self.M, self.Din = x.shape
        self.D = W2.shape[0]
        self.grad_scale = float(grad_scale)
        ws_bytes = L.lib().td_aligner_bwd_workspace_bytes(self.M, self.Din, self.D)
        self.ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=x.device)
        self.ws_bytes = ws_bytes

    def _call(self, phase, dW1, db1, dW2, db2, dg):
        L.launch_count += 4 if phase == L.BWD_NORM_W2 else 3
        L.check(
            L.lib().td_aligner_bwd(L.ptr(self.dy), L.dtype_code(self.dy), L.ptr(self.x), L.ptr(self.h0), L.ptr(self.h1),
                                   L.ptr(self.h2), L.ptr(self.rstd), L.ptr(self.W2), L.ptr(self.g), self.M, self.Din,
                                   self.D, self.grad_scale, L.ptr(dW1), L.ptr(db1), L.ptr(dW2), L.ptr(db2), L.ptr(dg),
                                   L.ptr(self.ws), self.ws_bytes, phase, L.stream_ptr()),
            "td_aligner_bwd",
        )

    def norm_and_linear2(self, dW2, db2, dg):
        self._call(L.BWD_NORM_W2, None, None, dW2, db2, dg)

    def gelu_and_linear1(self, dW1, db1):
        self._call(L.BWD_GELU_W1, dW1, db1, None, None, None)


def aligner_mse_fwd(x, W1, b1, W2, b2, g, eps: float, target, between_stages=None, target_row_index=None, defer_loss: bool = False):
    """Fused training forward against T5 targets: returns (loss, saved) with saved = (h0, h1, dh2, norm_partials), where
    dh2 / norm_partials are the T5LayerNorm backward of the MSE gradient for a unit upstream gradient (norm_partials = the
    per-CTA partial column sums for dg / db2, then the per-CTA loss partials). ``between_stages``: optional callable run after
    Linear1+GELU is enqueued and before anything reads W2 / b2. ``target_row_index`` (int64 [M]): row of ``target`` that belongs
    to each row of x. ``defer_loss``: leave the loss un-finished -- ``AlignerBackwardFromDh2(..., loss_out=loss)`` finishes it in
    the backward's own finisher launch (one launch fewer per training step)."""
    _need_cuda(x, W1, W2, g, target, target_row_index)
    M, Din = x.shape
    D = W1.shape[0]
    if target.dim() != 2 or target.shape[1] != D or (target_row_index is None and target.shape[0] != M):
        raise ValueError(f"target must be [{M}, {D}] (or indexed by target_row_index), got {tuple(target.shape)}")
    if target_row_index is not None and (target_row_index.dtype != torch.int64 or target_row_index.numel() != M):
        raise TypeError("target_row_index must be int64 [M]")
    dev = x.device
    h0 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
    h1 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
    dh2 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
    partials = torch.empty((L.lib().td_aligner_norm_partials_bytes(M, D),), dtype=torch.uint8, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    ws_bytes = L.lib().td_aligner_mse_fwd_workspace_bytes(M, Din, D)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.launch_count += 3 if defer_loss else 4
    extra = L.FWD_DEFER_LOSS if defer_loss else 0

    def call(stages):
        L.check(
            L.lib().td_aligner_mse_fwd(L.ptr(_contig(x, "x")), M, Din, D, L.ptr(W1), L.ptr(b1), L.ptr(W2), L.ptr(b2), L.ptr(g), eps,
                                       L.ptr(_contig(target, "target")), L.dtype_code(target), L.ptr(target_row_index), L.ptr(h0),
                                       L.ptr(h1), L.ptr(dh2), L.ptr(partials), L.ptr(loss), L.ptr(ws), ws_bytes, stages | extra, L.stream_ptr()),
            "td_aligner_mse_fwd",
        )

    if between_stages is None:
        call(3)
    else:
        call(1)
        between_stages()
        call(2)
    return loss, (h0, h1, dh2, partials)


class AlignerBackwardFromDh2:
    """Phased backward of the fused MSE path: everything is multiplied by grad_scale * upstream (a device scalar).
    One C call per method; inside a call the launch order is dh0 GEMM, ONE finisher launch (db1 | dg, db2 | loss), dW1 GEMM,
    dW2 GEMM. ``loss_out``: finish a loss deferred by ``aligner_mse_fwd(defer_loss=True)`` in the first finisher launch.
    ``stats`` (fp32 [2]): non-finite gradient counter (GradScaler); ``accumulate``: add into the gradient buffers."""

    def __init__(self, x, saved, W2, upstream, grad_scale: float = 1.0, loss_out=None, stats=None, accumulate: bool = False):
        self.x, (self.h0, self.h1, self.dh2, self.partials), self.W2 = x, saved, W2
        self.upstream = None if upstream is None else upstream.reshape(1).to(torch.float32).contiguous()
        self.M, self.Din = x.shape
        self.D = W2.shape[0]
        self.grad_scale = float(grad_scale)
        self.loss_out, self.stats, self.accumulate = loss_out, stats, bool(accumulate)
        self.ws_bytes = L.lib().td_aligner_bwd_workspace_bytes(self.M, self.Din, self.D)
        self.ws = torch.empty((self.ws_bytes,), dtype=torch.uint8, device=x.device)

    def _take_loss(self):
        lo, self.loss_out = self.loss_out, None  # finished by the first call that launches a finisher
        return lo

    def _count(self, phase):
        n = 0
        if phase & (L.BWD_GELU_W1 | L.BWD_GELU_ONLY):
            n += 2  # dh0 GEMM + finisher
        elif phase & (L.BWD_NORM_W2 | L.BWD_SMALL2_ONLY):
            n += 1  # finisher
        if phase & (L.BWD_GELU_W1 | L.BWD_W1_ONLY):
            n += 1
        if phase & (L.BWD_NORM_W2 | L.BWD_W2_ONLY):
            n += 1
        L.launch_count += n

    def _call(self, phase, dW1, db1, dW2, db2, dg):
        self._count(phase)
        loss_out = self._take_loss() if phase & (L.BWD_GELU_W1 | L.BWD_GELU_ONLY | L.BWD_NORM_W2 | L.BWD_SMALL2_ONLY) else None
        L.check(
            L.lib().td_aligner_bwd_dh2(L.ptr(self.dh2), L.ptr(self.x), L.ptr(self.h0), L.ptr(self.h1), L.ptr(self.W2),
                                       L.ptr(self.partials), self.M, self.Din, self.D, self.grad_scale,
                                       L.ptr(self.upstream), L.ptr(dW1), L.ptr(db1), L.ptr(dW2), L.ptr(db2), L.ptr(dg),
                                       L.ptr(loss_out), L.ptr(self.stats), int(self.accumulate),
                                       L.ptr(self.ws), self.ws_bytes, phase, L.stream_ptr()),
            "td_aligner_bwd_dh2",
        )

    def norm_and_linear2(self, dW2, db2, dg):
        self._call(L.BWD_NORM_W2, None, None, dW2, db2, dg)

    def gelu_and_linear1(self, dW1, db1):
        self._call(L.BWD_GELU_W1, dW1, db1, None, None, None)

    def gelu_linear1_and_small(self, dW1, db1, db2, dg):
        """dh0 GEMM, one finisher for all three small vectors (+ the deferred loss), dW1 GEMM."""
        self._call(L.BWD_GELU_W1 | L.BWD_SMALL2_ONLY, dW1, db1, None, db2, dg)

    def gelu_and_small(self, db1, db2, dg):
        """dh0 GEMM (dh0 stays in the workspace) and ONE finisher for all three small vectors (+ the deferred loss)."""
        self._call(L.BWD_GELU_ONLY | L.BWD_SMALL2_ONLY, None, db1, None, db2, dg)

    def norm_small(self, db2, dg):
        self._call(L.BWD_SMALL2_ONLY, None, None, None, db2, dg)

    def linear2_only(self, dW2):
        self._call(L.BWD_W2_ONLY, None, None, dW2, None, None)

    def _call_scatter(self, phase, dW1_dst, db1, dW2_dst, db2, dg, world, rank: int = -1, fold=None):
        self._count(phase)
        loss_out = self._take_loss() if phase & (L.BWD_GELU_W1 | L.BWD_GELU_ONLY | L.BWD_NORM_W2 | L.BWD_SMALL2_ONLY) else None
        L.check(
            L.lib().td_aligner_bwd_dh2_scatter(L.ptr(self.dh2), L.ptr(self.x), L.ptr(self.h0), L.ptr(self.h1), L.ptr(self.W2),
                                               L.ptr(self.partials), self.M, self.Din, self.D, self.grad_scale,
                                               L.ptr(self.upstream), dW1_dst, L.ptr(db1), dW2_dst, L.ptr(db2), L.ptr(dg),
                                               L.ptr(loss_out), L.ptr(self.stats), world, int(rank),
                                               None if fold is None else C.cast(C.pointer(fold), C.c_void_p),
                                               L.ptr(self.ws), self.ws_bytes, phase, L.stream_ptr()),
            "td_aligner_bwd_dh2_scatter",
        )

    def gelu_linear1_small_scatter(self, dW1_dst, db1, db2, dg, world: int, rank: int = -1):
        """As ``gelu_linear1_and_small`` with dW1's rows stored to their owner ranks (``dW1_dst``: host array of ``world``
        device pointers). ``rank`` (of the caller, >= 0) turns on the rank-rotated tile order of the scattered GEMMs."""
        self._call_scatter(L.BWD_GELU_W1 | L.BWD_SMALL2_ONLY, dW1_dst, db1, None, db2, dg, world, rank)

    def gelu_and_small_scatter(self, db1, db2, dg, world: int, fold):
        """As ``gelu_and_small`` in the peer data-parallel step: the finisher also stores the three small vectors into this rank's
        slot at every rank (``fold``: a ``PeerFold`` with ``small_dst``)."""
        self._call_scatter(L.BWD_GELU_ONLY | L.BWD_SMALL2_ONLY, None, db1, None, db2, dg, world, -1, fold)

    def linear1_only_scatter(self, dW1_dst, world: int, rank: int = -1, fold=None):
        """dW1 GEMM from the dh0 a ``gelu_and_small`` call left in the workspace, rows stored to their owner ranks. ``fold`` (a
        ``PeerFold`` with ``signal_flags``): the GEMM bumps that counter at every rank once all of its stores have completed."""
        self._call_scatter(L.BWD_W1_ONLY, dW1_dst, None, None, None, None, world, rank, fold)

    def linear2_only_scatter(self, dW2_dst, world: int, rank: int = -1, fold=None):
        self._call_scatter(L.BWD_W2_ONLY, None, None, dW2_dst, None, None, world, rank, fold)


def rmsnorm_fwd(x: torch.Tensor, g: torch.Tensor, eps: float = 1e-6, out_bf16: bool = False):
    _need_cuda(x, g)
    M, D = x.shape
    y = torch.empty((M, D), dtype=torch.bfloat16 if out_bf16 else torch.float32, device=x.device)
    rstd = torch.empty((M,), dtype=torch.float32, device=x.device)
    L.launch_count += 1
    L.check(L.lib().td_rmsnorm_fwd(L.ptr(_contig(x, "x")), L.ptr(g), eps, M, D, L.ptr(y), L.BF16 if out_bf16 else L.F32,
                                   L.ptr(rstd), L.stream_ptr()), "td_rmsnorm_fwd")
    return y, rstd


def rmsnorm_bwd(dy, x, rstd, g):
    _need_cuda(dy, x, rstd, g)
    M, D = x.shape
    dx = torch.empty((M, D), dtype=torch.bfloat16, device=x.device)
    dg = torch.empty((D,), dtype=torch.float32, device=x.device)
    dxsum = torch.empty((D,), dtype=torch.float32, device=x.device)
    ws_bytes = L.lib().td_rmsnorm_bwd_workspace_bytes(M, D)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=x.device)
    L.launch_count += 3
    L.check(L.lib().td_rmsnorm_bwd(L.ptr(_contig(dy, "dy")), L.dtype_code(dy), L.ptr(x), L.ptr(rstd), L.ptr(g), M, D,
                                   L.ptr(dx), L.ptr(dg), L.ptr(dxsum), L.ptr(ws), ws_bytes, L.stream_ptr()), "td_rmsnorm_bwd")
    return dx, dg, dxsum


def gemm_workspace(device, stream_k: bool = True):
    """(tensor, nbytes) workspace for the stream-K tail of one GEMM launch; (None, 0) disables the tail."""
    if not stream_k:
        return None, 0
    n = L.lib().td_gemm_workspace_bytes()
    return torch.empty((n,), dtype=torch.uint8, device=device), n


def linear_bf16(x, W, bias=None, stream_k: bool = True):
    _need_cuda(x, W)
    M, K = x.shape
    N = W.shape[0]
    out = torch.empty((M, N), dtype=torch.bfloat16, device=x.device)
    ws, ws_bytes = gemm_workspace(x.device, stream_k)
    L.launch_count += 1
    L.check(L.lib().td_linear_bf16(L.ptr(_contig(x, "x")), M, K, L.ptr(_contig(W, "W")), N, L.ptr(bias), L.ptr(out),
                                   L.ptr(ws), ws_bytes, L.stream_ptr()), "td_linear_bf16")
    return out


def linear_bf16_dx(dy, W, stream_k: bool = True):
    """Input gradient of ``linear_bf16`` for a frozen weight: dy [M, N] bf16, W [N, K] bf16 (nn.Linear layout) -> dx [M, K] bf16.
    W is contracted over its row index and read in place (MN-major tensor-core operand)."""
    _need_cuda(dy, W)
    M, N = dy.shape
    if W.shape[0] != N or dy.dtype != torch.bfloat16 or W.dtype != torch.bfloat16:
        raise TypeError("linear_bf16_dx: dy [M, N] and W [N, K] must be bfloat16")
    K = W.shape[1]
    dx = torch.empty((M, K), dtype=torch.bfloat16, device=dy.device)
    ws, ws_bytes = gemm_workspace(dy.device, stream_k)
    L.launch_count += 1
    L.check(L.lib().td_linear_bf16_dx(L.ptr(_contig(dy, "dy")), M, N, L.ptr(_contig(W, "W")), K, L.ptr(dx), L.ptr(ws), ws_bytes,
                                      L.stream_ptr()), "td_linear_bf16_dx")
    return dx


def gemm_f32out(A, B, a_mn_major: bool, b_mn_major: bool, alpha: float = 1.0, cta_pair: bool = True, stream_k: bool = True,
                out=None):
    """Test entry: D[M, N] fp32 = alpha * A.B^T; K-major operand = [rows, K], MN-major operand = [K, rows].
    ``out``: accumulate into this tensor instead of returning a fresh one."""
    _need_cuda(A, B)
    M, K = (A.shape[1], A.shape[0]) if a_mn_major else A.shape
    N = B.shape[1] if b_mn_major else B.shape[0]
    accumulate = out is not None
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    ws, ws_bytes = gemm_workspace(A.device, stream_k)
    L.launch_count += 1
    for t, n in ((A, "A"), (B, "B")):  # a column slice of a K-major operand is fine: TMA only needs the row pitch
        if t.dim() != 2 or t.stride(1) != 1:
            raise ValueError(f"{n} must be 2-D with unit inner stride")
    L.check(L.lib().td_gemm_bf16_f32out(L.ptr(A), A.stride(0), int(a_mn_major), L.ptr(B),
                                        B.stride(0), int(b_mn_major), M, N, K, alpha, L.ptr(out), int(cta_pair), int(accumulate),
                                        L.ptr(ws), ws_bytes, L.stream_ptr()), "td_gemm_bf16_f32out")
    return out


# ------------------------------------------------------------------------------------------------ losses
def masked_mse_fwd_bwd(y, target, row_mask=None, grad_scale: float = 1.0, want_grad: bool = True):
    """Returns (loss fp32 scalar tensor, dy or None). y, target [M, D] float32/bfloat16; row_mask int64 [M] or None."""
    _need_cuda(y, target, row_mask)
    M, D = y.shape
    if target.shape != y.shape:
        raise ValueError("target shape must match y")
    if row_mask is not None and (row_mask.dtype != torch.int64 or row_mask.numel() != M):
        raise TypeError("row_mask must be int64 [M]")
    loss = torch.empty((), dtype=torch.float32, device=y.device)
    dy = torch.empty_like(y) if want_grad else None
    ws_bytes = L.lib().td_loss_workspace_bytes(M)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=y.device)
    L.launch_count += 3
    L.check(L.lib().td_masked_mse_fwd_bwd(L.ptr(_contig(y, "y")), L.dtype_code(y), L.ptr(_contig(target, "target")),
                                          L.dtype_code(target), L.ptr(row_mask), M, D, grad_scale, L.ptr(loss), L.ptr(dy),
                                          L.ptr(ws), ws_bytes, L.stream_ptr()), "td_masked_mse_fwd_bwd")
    return loss, dy


def masked_ce_fwd_bwd(logits, labels, grad_scale: float = 1.0, want_grad: bool = True):
    """CrossEntropyLoss(ignore_index=-100) forward + dlogits. logits [R, V] float32/bfloat16, labels int64 [R]."""
    _need_cuda(logits, labels)
    R, V = logits.shape
    if labels.dtype != torch.int64 or labels.numel() != R:
        raise TypeError("labels must be int64 [R]")
    loss = torch.empty((), dtype=torch.float32, device=logits.device)
    dz = torch.empty_like(logits) if want_grad else None
    ws_bytes = L.lib().td_loss_workspace_bytes(R)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=logits.device)
    L.launch_count += 3
    L.check(L.lib().td_masked_ce_fwd_bwd(L.ptr(_contig(logits, "logits")), L.dtype_code(logits), L.ptr(_contig(labels, "labels")),
                                         R, V, grad_scale, L.ptr(loss), L.ptr(dz), L.ptr(ws), ws_bytes, L.stream_ptr()),
            "td_masked_ce_fwd_bwd")
    return loss, dz


def lm_head_ce(seq, W_lm, labels, grad_scale: float = 1.0, want_grad: bool = True, keep_logits: bool = False):
    """Frozen T5 output head + loss (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:236-246 under bf16 autocast) and their
    backward down to the decoder output: seq [R, K] bf16, W_lm [V, K] bf16, labels int64 [R] (-100 = ignore).
    Returns (loss fp32 scalar, dseq [R, K] bf16 or None, logits [R, V] bf16 or None). Unless ``keep_logits``, the gradient of the
    logits overwrites them in place (one [R, V] buffer instead of two)."""
    _need_cuda(seq, W_lm, labels)
    R, K = seq.shape
    V = W_lm.shape[0]
    if seq.dtype != torch.bfloat16 or W_lm.dtype != torch.bfloat16 or W_lm.shape[1] != K:
        raise TypeError("lm_head_ce: seq [R, K] and W_lm [V, K] must be bfloat16")
    if labels.dtype != torch.int64 or labels.numel() != R:
        raise TypeError("labels must be int64 [R]")
    dev = seq.device
    logits = torch.empty((R, V), dtype=torch.bfloat16, device=dev)
    dlogits = None
    if want_grad:
        dlogits = torch.empty_like(logits) if keep_logits else logits
    dseq = torch.empty((R, K), dtype=torch.bfloat16, device=dev) if want_grad else None
    loss = torch.empty((), dtype=torch.float32, device=dev)
    ws_bytes = L.lib().td_lm_head_ce_workspace_bytes(R)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.launch_count += 5 if want_grad else 4
    L.check(L.lib().td_lm_head_ce_fwd_bwd(L.ptr(_contig(seq, "seq")), R, K, L.ptr(_contig(W_lm, "W_lm")), V, L.ptr(_contig(labels, "labels")),
                                          grad_scale, L.ptr(loss), L.ptr(logits), L.ptr(dlogits), L.ptr(dseq), L.ptr(ws), ws_bytes,
                                          L.stream_ptr()), "td_lm_head_ce_fwd_bwd")
    return loss, dseq, (logits if keep_logits or not want_grad else None)



# ------------------------------------------------------------------------------------------------ T5 attention (8 f-1)
def _rows_operand(t, name, inner):
    """A [rows, >= inner] bf16 operand with unit inner stride and a row pitch that is a multiple of 8 (column slices allowed)."""
    if t.dtype != torch.bfloat16 or t.dim() != 2 or t.shape[1] != inner:
        raise TypeError(f"{name} must be a bfloat16 [rows, {inner}] tensor, got {t.dtype} {tuple(t.shape)}")
    if t.stride(1) != 1 or t.stride(0) % 8 or t.stride(0) < inner:
        raise ValueError(f"{name} must have unit column stride and a row pitch that is a multiple of 8 (stride {t.stride()})")
    return t


def _attn_common(q, k, v, cu_q, cu_k, n_heads, bias_by_distance):
    _need_cuda(q, k, v, cu_q, cu_k, bias_by_distance)
    inner = q.shape[1]
    for t, n in ((q, "q"), (k, "k"), (v, "v")):
        _rows_operand(t, n, inner)
    if k.shape[0] != v.shape[0]:
        raise ValueError("k and v must have the same rows")
    if cu_q.dtype != torch.int32 or (cu_k is not None and (cu_k.dtype != torch.int32 or cu_k.numel() != cu_q.numel())):
        raise TypeError("cu_q / cu_k must be int32 [B + 1]")
    self_attention = bias_by_distance is not None
    n_dist = 0
    if self_attention:
        if bias_by_distance.dtype != torch.float32 or bias_by_distance.dim() != 2 or bias_by_distance.shape[0] != n_heads:
            raise TypeError(f"bias_by_distance must be float32 [{n_heads}, n_dist]")
        _contig(bias_by_distance, "bias_by_distance")
        if cu_k is not None and cu_k.data_ptr() != cu_q.data_ptr():
            raise ValueError("self-attention attends to its own rows: pass cu_k=None or cu_q")
        cu_k = None
        n_dist = bias_by_distance.shape[1]
    elif cu_k is None:
        raise ValueError("cross-attention needs cu_k")
    return inner, self_attention, cu_k, n_dist


def t5_attention_fwd(q, k, v, cu_q, cu_k, max_len_q: int, max_len_k: int, n_heads: int, bias_by_distance=None, o=None,
                     need_lse: bool = True):
    """T5 attention core on packed rows (no 1/sqrt(d_kv) scaling, fp32 softmax, d_kv = 64): sample b's queries are rows
    ``cu_q[b]:cu_q[b+1]`` of ``q [Mq, 64 H]``, its keys / values rows ``cu_k[b]:cu_k[b+1]`` of ``k`` / ``v [Mk, 64 H]``.
    ``bias_by_distance`` ([H, n_dist] fp32, see ``t5.t5_position_bias_by_distance``) selects causal self-attention (keys = the
    query rows, ``cu_k`` None or ``cu_q``). Inputs may be column slices of a fused projection output. ``max_len_*`` bound the
    samples' lengths (host-known; no device sync). Returns ``(o [Mq, 64 H] bf16, lse [H, Mq] fp32 or None)``; ``o`` may be given."""
    inner, self_attention, cu_k, n_dist = _attn_common(q, k, v, cu_q, cu_k, n_heads, bias_by_distance)
    Mq = q.shape[0]
    if o is None:
        o = torch.empty((Mq, inner), dtype=torch.bfloat16, device=q.device)
    _rows_operand(o, "o", inner)
    lse = torch.empty((n_heads, Mq), dtype=torch.float32, device=q.device) if need_lse else None
    L.launch_count += 1
    L.check(L.lib().td_t5_attention_fwd(L.ptr(q), q.stride(0), L.ptr(k), k.stride(0), L.ptr(v), v.stride(0), L.ptr(cu_q), L.ptr(cu_k),
                                        cu_q.numel() - 1, n_heads, inner, int(max_len_q), int(max_len_k), Mq, int(self_attention),
                                        L.ptr(bias_by_distance), n_dist, L.ptr(o), o.stride(0), L.ptr(lse), L.stream_ptr()),
            "td_t5_attention_fwd")
    return o, lse


def t5_attention_bwd(dout, q, k, v, o, lse, cu_q, cu_k, max_len_q: int, max_len_k: int, n_heads: int, bias_by_distance=None,
                     dq=None, dk=None, dv=None):
    """Backward of ``t5_attention_fwd``: returns ``(dq, dk, dv)`` bf16. Any of them may be given, e.g. ``dk`` / ``dv`` as the two
    column halves of one ``[Mk, 2 inner]`` buffer -- the input gradient of a fused ``[Wk; Wv]`` projection. Three launches
    (row sums of dO * O, dK / dV, dQ); deterministic."""
    inner, self_attention, cu_k, n_dist = _attn_common(q, k, v, cu_q, cu_k, n_heads, bias_by_distance)
    Mq, Mk = q.shape[0], k.shape[0]
    _need_cuda(dout, o, lse)
    _rows_operand(dout, "dout", inner)
    _rows_operand(o, "o", inner)
    if lse is None or lse.dtype != torch.float32 or tuple(lse.shape) != (n_heads, Mq):
        raise TypeError(f"lse must be float32 [{n_heads}, {Mq}] (run the forward with need_lse=True)")
    _contig(lse, "lse")
    dev = q.device
    dq = torch.empty((Mq, inner), dtype=torch.bfloat16, device=dev) if dq is None else dq
    dk = torch.empty((Mk, inner), dtype=torch.bfloat16, device=dev) if dk is None else dk
    dv = torch.empty((Mk, inner), dtype=torch.bfloat16, device=dev) if dv is None else dv
    for t, n in ((dq, "dq"), (dk, "dk"), (dv, "dv")):
        _rows_operand(t, n, inner)
    ws_bytes = L.lib().td_t5_attention_workspace_bytes(Mq, n_heads)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.launch_count += 3
    L.check(L.lib().td_t5_attention_bwd(L.ptr(dout), dout.stride(0), L.ptr(q), q.stride(0), L.ptr(k), k.stride(0), L.ptr(v), v.stride(0),
                                        L.ptr(cu_q), L.ptr(cu_k), cu_q.numel() - 1, n_heads, inner, int(max_len_q), int(max_len_k), Mq,
                                        int(self_attention), L.ptr(bias_by_distance), n_dist, L.ptr(o), o.stride(0), L.ptr(lse),
                                        L.ptr(dq), dq.stride(0), L.ptr(dk), dk.stride(0), L.ptr(dv), dv.stride(0), L.ptr(ws), ws_bytes,
                                        L.stream_ptr()), "td_t5_attention_bwd")
    return dq, dk, dv


# ------------------------------------------------------------------------------------------------ T5 gated-GELU FFN (8 f-1)
def _ffn_dims(x, wi, wo, ln_w):
    _need_cuda(x, wi, wo, ln_w)
    M, d = x.shape
    d_ff = wo.shape[1]
    if x.dtype != torch.bfloat16 or wi.dtype != torch.bfloat16 or wo.dtype != torch.bfloat16 or ln_w.dtype != torch.float32:
        raise TypeError("t5_ffn: x, wi, wo must be bfloat16 and ln_w float32")
    if tuple(wi.shape) != (2 * d_ff, d) or tuple(wo.shape) != (d, d_ff) or tuple(ln_w.shape) != (d,):
        raise ValueError(f"t5_ffn: need wi [2 d_ff, d], wo [d, d_ff], ln_w [d]; got {tuple(wi.shape)}, {tuple(wo.shape)}, {tuple(ln_w.shape)}")
    for t, n in ((x, "x"), (wi, "wi"), (wo, "wo"), (ln_w, "ln_w")):
        _contig(t, n)
    return M, d, d_ff


def t5_ffn_fwd(x, wi, wo, ln_w, eps: float, want_ab: bool = True, want_gated: bool = False):
    """T5LayerFF (gated-GELU) forward on packed rows: ``x [M, d]`` bf16, ``wi [2 d_ff, d]`` bf16 with wi_0 / wi_1 interleaved in
    blocks of 32 rows (``t5.T5FeedForwardWeights``), ``wo [d, d_ff]`` bf16, ``ln_w [d]`` fp32. Returns ``(out [M, d] bf16, rstd [M]
    fp32, ab [M, 2 d_ff] bf16 or None, gated [M, d_ff] bf16 or None)``: ``ab`` (a / b in wi's interleaved column order) is what the
    backward needs; ``want_ab=False`` is the inference path. Three launches."""
    M, d, d_ff = _ffn_dims(x, wi, wo, ln_w)
    dev = x.device
    out = torch.empty((M, d), dtype=torch.bfloat16, device=dev)
    rstd = torch.empty((M,), dtype=torch.float32, device=dev)
    ab = torch.empty((M, 2 * d_ff), dtype=torch.bfloat16, device=dev) if want_ab else None
    gated = torch.empty((M, d_ff), dtype=torch.bfloat16, device=dev) if want_gated else None
    ws_bytes = L.lib().td_t5_ffn_workspace_bytes(M, d, d_ff)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.launch_count += 3
    L.check(L.lib().td_t5_ffn_fwd(L.ptr(x), M, d, d_ff, L.ptr(ln_w), eps, L.ptr(wi), L.ptr(wo), L.ptr(out), L.ptr(rstd), L.ptr(ab),
                                  L.ptr(gated), L.ptr(ws), ws_bytes, L.stream_ptr()), "td_t5_ffn_fwd")
    return out, rstd, ab, gated


def t5_ffn_bwd(dy, x, rstd, ab, wi, wo, ln_w, want_d_ab: bool = False):
    """Input gradient of ``t5_ffn_fwd`` (frozen weights): ``dy [M, d]`` bf16 and the forward's ``x``, ``rstd``, ``ab``. Returns
    ``(dx [M, d] bf16, d_ab [M, 2 d_ff] bf16 or None)``; ``d_ab`` holds dL/da and dL/db in wi's interleaved column order. Three
    launches; deterministic."""
    M, d, d_ff = _ffn_dims(x, wi, wo, ln_w)
    _need_cuda(dy, rstd, ab)
    if dy.dtype != torch.bfloat16 or tuple(dy.shape) != (M, d):
        raise TypeError(f"t5_ffn_bwd: dy must be bfloat16 [{M}, {d}]")
    if ab is None or ab.dtype != torch.bfloat16 or tuple(ab.shape) != (M, 2 * d_ff):
        raise TypeError(f"t5_ffn_bwd: ab must be the forward's bfloat16 [{M}, {2 * d_ff}] (run it with want_ab=True)")
    if rstd.dtype != torch.float32 or rstd.numel() != M:
        raise TypeError(f"t5_ffn_bwd: rstd must be float32 [{M}]")
    for t, n in ((dy, "dy"), (ab, "ab"), (rstd, "rstd")):
        _contig(t, n)
    dev = x.device
    dx = torch.empty((M, d), dtype=torch.bfloat16, device=dev)
    d_ab = torch.empty((M, 2 * d_ff), dtype=torch.bfloat16, device=dev) if want_d_ab else None
    ws_bytes = L.lib().td_t5_ffn_workspace_bytes(M, d, d_ff)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.launch_count += 3
    L.check(L.lib().td_t5_ffn_bwd(L.ptr(dy), L.ptr(x), L.ptr(rstd), L.ptr(ln_w), L.ptr(ab), L.ptr(wi), L.ptr(wo), M, d, d_ff, L.ptr(dx),
                                  L.ptr(d_ab), L.ptr(ws), ws_bytes, L.stream_ptr()), "td_t5_ffn_bwd")
    return dx, d_ab
