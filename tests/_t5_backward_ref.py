"""Float64 staged reference of the T5 objective's backward, for per-element parity at Flan-T5-XXL width (d 4096, H 64, d_ff 10240,
V 32128): the output head with its cross-entropy, the attention core in both directions, and the input gradients of the three decoder
sublayers. Test infrastructure only; the product path never imports it.

As in ``_aligner_step_ref`` (whose ``bf16``, ``ulp``, ``product``, ``contract_rows``, ``gemm_error``, ``ACC``, ``RUN_SUM`` and ``ROW_EPS``
this builds on), every stage takes the kernels' own outputs of the stage before it, so errors do not compound and each bound can be
tight. Each function returns the exact float64 result together with a per-element bound on the error of the kernel's fp32
arithmetic; the caller adds the rounding of the output (half a bf16 ulp, or one ulp where the kernel rounds twice).

Stages and their rounding points (header include/thinkdiff_b200.h, csrc/rowops_sm100.cuh, csrc/attn_sm100.cuh):

    logits  = bf16(seq W^T)                                            (K = 4096)
    dlogits = bf16(2^(z log2e + log2(gs / sum) - m) - gs [label])      gs = grad_scale / n_valid; ignored rows exactly 0
    loss    = sum_rows (log(sum) + m ln2 - z[label]) / n_valid         all fp32
    dseq    = bf16(dlogits W)                                          (K = 32128)
    attention forward:   O = bf16(sum_j bf16(p_j) v_j / l), l = sum_j p_j, p_j = 2^((s_j - m) log2e), lse = m + log l
    attention backward:  P = 2^((s - lse) log2e), Delta = rowsum(dO o O), dS = bf16(P (dO V^T - Delta)),
                         dV = bf16(bf16(P)^T dO), dK = bf16(dS^T Q), dQ = bf16(dS K)
    FFN:                 t = bf16(dy wo), d_a = bf16(bf16(t b) gelu_new'(a)), d_b = bf16(t bf16(gelu_new(a))), dxn = bf16(d_ab wi)
    every sublayer:      dx = bf16(dy + rstd g dxn - x rstd^3 mean(g dxn x))   with the forward's rstd

Everything is float64 torch arithmetic on whatever device the inputs live on. tests/test_t5_backward_ref_cpu.py pins these functions
on the CPU to ``_t5_attention_ref.attention_packed`` under autograd, ``oracle.t5_head_ref``, ``_t5_ffn_ref`` and
``_t5_decoder_block_ref``.
"""
from __future__ import annotations

import math

import torch

from _aligner_step_ref import ACC, BLOCK_ROWS, ROW_EPS, bf16, contract_rows, ulp
from thinkdiff_mlre_b200.t5 import interleave_pairs, split_pairs

U = 2.0 ** -24  # fp32 unit roundoff
LOG2E = 1.0 / math.log(2.0)
# bf16 unit roundoff: the relative error of rounding P (forward and dK/dV) and dS to bf16 before their MMAs. The forward sums l from
# the unrounded p, so the rounding of P reaches O undivided: 2^-8 (P |V|)
PROB = 2.0 ** -8
# ex2.approx.f32 (MUFU.EX2): at most 2 fp32 ulp relative (PTX ISA), i.e. 2^-22
EX2 = 2.0 ** -22
# the exponent argument fmaf(s, log2e, -m log2e) in fp32: kLog2e's own rounding, the rounding of m log2e and of the fma, each at most
# 2^-24 of log2e (|s| + |m|); back in natural units (times ln 2) and with the fp32 bias add: below 2^-22 (|s| + |m|)
ARG = 2.0 ** -22
# ex2.approx.ftz flushes results below 2^-126 to zero, and the tensor core flushes fp32 subnormals: an absolute error of up to 2^-126
# on every probability, every dS formed from one and every attention output (far below any output's ulp unless the output itself is
# that small, e.g. dK of a key whose every probability is below 2^-100)
FTZ = 2.0 ** -126
# gelu_tanh / gelu_tanh' in the FFN's epilogue (ptx_sm100.cuh gelu_tanh_gate): u = C (x + 0.044715 x^3) carries four fp32 roundings,
# so e = ex2(-2 log2e |u|) is off by 2 |u| 5 2^-24 relative beside ex2's own 2^-22; rcp adds 2^-22, the products 2^-24 each. s = r or
# e r within 2^-20 (1 + |u|) of sigmoid(2u), ds = 2 e r^2 C (1 + 3 c x^2) within twice that
GELU_TANH_REL = 2.0 ** -20
ATTN_TILE = 128


# ------------------------------------------------------------------------------------------------ GEMMs contracting a long K
def contract(a: torch.Tensor, w: torch.Tensor):
    """(a w, bound) for a [M, K], w [K, N] (a linear layer's input gradient, K up to 32128): ``contract_rows`` over K, so the bound
    carries the fp32 ulp of the running partial sum per MMA accumulation beside ACC |a| |w|."""
    return contract_rows(a.T, w)


# ------------------------------------------------------------------------------------------------ cross-entropy
def ce_rows(z: torch.Tensor, labels: torch.Tensor, grad_scale: float, n_valid: int) -> dict:
    """CrossEntropyLoss(ignore_index=-100) of the kernel's bf16 logits ``z [r, V]``, in float64, per row:

      loss_row = logsumexp(z) - z[label] (0 on ignored rows), dz = (softmax(z) - onehot) grad_scale / n_valid (0 on ignored rows),
      dz_arith: a bound on the error of masked_ce_kernel's fp32 arithmetic in dz, and loss_arith: the same for loss_row.

    The kernel forms p gs as one exp2f of fmaf(z, log2e, shift), shift = -m + log2f(gs / sum), m = max(z) log2e, and subtracts gs at the
    label. The exponent argument is off by at most 2^-22 (2 |z|max log2e + |log2(gs / sum)| + 1) (four fp32 roundings and log2f's
    2 ulp); exp2f adds 2 ulp; the sum of the exponentials is off by (V / 256 + 32) 2^-24 relative (each thread adds V / 256 terms in
    order, then two five-level shuffle trees) plus the error of its terms. Together a relative error ``rel`` of p gs; at the label,
    where p - 1 cancels, that is an absolute error rel p gs, which is why the bound is written as rel p |gs| on every element.
    loss_row = logf(sum) + m ln 2 - z[label]: the sum's relative error, logf's and the two roundings' 2^-22 (|log sum| + |z|max + |row|)."""
    z = z.to(torch.float64)
    V = z.shape[1]
    valid = labels != -100
    lab = labels.clamp(0, V - 1)
    lse = torch.logsumexp(z, 1)
    p = torch.exp(z - lse[:, None])
    zl = z.gather(1, lab[:, None]).squeeze(1)
    gs = grad_scale / n_valid
    zmax = z.abs().amax(1)
    log_sum = lse - z.amax(1)
    arg = 2.0 ** -22 * (2 * zmax * LOG2E + (math.log2(abs(gs)) - log_sum * LOG2E).abs() + 1)
    sum_rel = (V / 256 + 32) * U + math.log(2.0) * arg + EX2
    rel = 2 * (math.log(2.0) * arg + EX2) + sum_rel + U  # + gs = grad_scale / n_valid in fp32
    dz = p * gs
    dz.scatter_add_(1, lab[:, None], torch.full_like(zl[:, None], -gs))
    dz = torch.where(valid[:, None], dz, 0.0)
    dz_arith = torch.where(valid[:, None], rel[:, None] * p * abs(gs), 0.0)
    row = torch.where(valid, lse - zl, 0.0)
    row_arith = torch.where(valid, sum_rel + 2.0 ** -22 * (log_sum.abs() + zmax + row.abs() + 1), 0.0)
    return {"loss_row": row, "loss_arith": row_arith, "dz": dz, "dz_arith": dz_arith}


def dlogits_error(value: torch.Tensor, ce: dict):
    """(|error|, tolerance) of the kernel's bf16 dlogits: the output rounding (half an ulp) and the fp32 arithmetic below one more
    half ulp on every element (within one bf16 ulp), plus the absolute fp32 term on the label's element. Ignored rows: exactly 0."""
    v = value.to(torch.float64)
    ref = ce["dz"]
    tol = torch.where(ce["dz_arith"] > 0, ulp(torch.maximum(v.abs(), ref.abs())) + ce["dz_arith"], 0.0)
    return (v - ref).abs(), tol


def loss_tolerance(row_arith_sum: float, row_abs_sum: float, R: int, n_valid: int) -> float:
    """loss_finish_kernel sums the R fp32 row losses (R / 256 in order per thread, then two five-level trees) and divides by n_valid:
    (R / 256 + 16) 2^-24 of the sum of |row| beside the rows' own error, over n_valid."""
    return (row_arith_sum + (R / 256 + 16) * U * row_abs_sum) / n_valid


# ------------------------------------------------------------------------------------------------ attention core
def _heads(x: torch.Tensor, H: int) -> torch.Tensor:
    return x.to(torch.float64).reshape(x.shape[0], H, x.shape[1] // H).transpose(0, 1)  # [H, L, 64]


def _packed(x: torch.Tensor) -> torch.Tensor:
    return x.transpose(0, 1).reshape(x.shape[1], x.shape[0] * x.shape[2])


def scores(qh, kh, bias_by_distance=None, mutate: str | None = None, drop_last_tile: bool = False):
    """S [H, T, L] in float64 (masked: -inf) and the bound ACC |q| |k|^T on the fp32 MMA that forms it. Causal self-attention with
    ``bias_by_distance`` [H, n_dist]: bias min(i - j, n_dist - 1). ``mutate`` builds deliberately wrong references for the checks that
    show the bounds can fail: "mask" lets query i see key i + 1, "bias" reads the bias at min(i - j + 1, n_dist - 1);
    ``drop_last_tile`` leaves out the sample's last 128-key tile."""
    s = qh @ kh.transpose(1, 2)
    eps = ACC * (qh.abs() @ kh.abs().transpose(1, 2))
    T, L = s.shape[1], s.shape[2]
    if bias_by_distance is not None:
        n = torch.arange(T, device=s.device)[:, None] - torch.arange(L, device=s.device)[None, :]
        nd = bias_by_distance.shape[1]
        s = s + bias_by_distance.to(torch.float64)[:, (n + (mutate == "bias")).clamp(0, nd - 1)]
        s = s.masked_fill(n < -(mutate == "mask"), float("-inf"))
    if drop_last_tile and L > ATTN_TILE:
        s[..., (L - 1) // ATTN_TILE * ATTN_TILE :] = float("-inf")
    return s, eps


def _finite(t, mask):
    return torch.where(mask, t, 0.0)


def attention_sample(q, k, v, H: int, bias_by_distance=None, o_k=None, lse_k=None, dout=None, mutate=None, drop_last_tile=False) -> dict:
    """One sample of the attention core in float64: q [T, 64 H], k / v [L, 64 H] (bf16 values), heads in column blocks of 64.

    Forward: O, lse and their bounds ``o_arith`` / ``lse_arith``. The kernel rounds the unnormalised p to bf16 before P.V while it sums
    l from the unrounded values: PROB (P |V|). Each p is off by FTZ plus a relative delta = eps + ARG (|s| + 2 |s|max) + n_kt EX2 from the score's
    accumulation, the exponent argument (the running max and the rescale alpha = 2^((m_old - m) log2e) included) and one ex2 per key
    tile; weights off by delta move O by at most sum_j P_j delta_j (|v_j| + |O|). l is summed in fp32 (127 additions per tile and the
    rescale per tile: (128 + 2 n_kt) 2^-24), P.V accumulates in the tensor core (ACC).

    Backward (``dout`` given), staged on the kernel's ``o_k`` / ``lse_k`` (default: the reference's own): P = exp(S - lse_k),
    Delta = rowsum(dO o O_k), dS = P (dP - Delta). P is off by P (eps + ARG (|s| + |lse_k|) + EX2) + FTZ, dP by ACC |dO| |V|^T, Delta by
    ACC sum |dO o O_k|; dS is rounded to bf16 before its MMAs (PROB |dS|), P before dV's (PROB P). dV, dK, dQ add ACC of their own
    contraction. Returns packed [rows, 64 H] tensors (lse [H, T]) and ``*_arith`` bounds; the output's half ulp is the caller's."""
    qh, kh, vh = _heads(q, H), _heads(k, H), _heads(v, H)
    s, eps = scores(qh, kh, bias_by_distance, mutate, drop_last_tile)
    T, L = s.shape[1], s.shape[2]
    vis = torch.isfinite(s)
    n_kt = -(-L // ATTN_TILE)
    out = {}
    if L == 0:  # no keys: O = 0 and dQ = 0 exactly, lse = -inf
        z = torch.zeros_like(q, dtype=torch.float64)
        out.update(o=z, o_arith=z, lse=torch.full((H, T), float("-inf"), dtype=torch.float64, device=q.device),
                   lse_arith=torch.zeros((H, T), dtype=torch.float64, device=q.device))
        if dout is not None:
            zk = torch.zeros_like(k, dtype=torch.float64)
            out.update(dq=z, dq_arith=z, dk=zk, dk_arith=zk, dv=zk, dv_arith=zk)
        return out
    lse = torch.logsumexp(s, -1)
    sabs = _finite(s.abs(), vis)
    smax = sabs.amax(-1, keepdim=True)
    P = _finite(torch.exp(s - lse[..., None]), vis)
    o = P @ vh
    delta = _finite(eps + ARG * (sabs + 2 * smax) + n_kt * EX2, vis)
    Pd = P * delta + FTZ * vis
    l_sum = (ATTN_TILE + 2 * n_kt) * U
    o_arith = (PROB + ACC + l_sum) * (P @ vh.abs()) + Pd @ vh.abs() + Pd.sum(-1, keepdim=True) * o.abs()
    lse_arith = Pd.sum(-1) + l_sum + 2.0 ** -22 * (lse.abs() + smax.squeeze(-1) + 8)
    out.update(o=_packed(o), o_arith=_packed(o_arith), lse=lse, lse_arith=lse_arith)
    if dout is None:
        return out
    ok = o if o_k is None else _heads(o_k, H)
    lk = lse if lse_k is None else lse_k.to(torch.float64)
    dOh = _heads(dout, H)
    Pb = _finite(torch.exp(s - lk[..., None]), vis)
    dP = dOh @ vh.transpose(1, 2)
    Dl = (dOh * ok).sum(-1, keepdim=True)
    dS = Pb * (dP - Dl)
    e_P = Pb * _finite(eps + ARG * (sabs + lk.abs()[..., None]) + EX2, vis) + FTZ * vis
    e_dS = ((PROB + ACC) * dS.abs() + e_P * (dP - Dl).abs() + FTZ * vis
            + Pb * ACC * (dOh.abs() @ vh.abs().transpose(1, 2) + (dOh.abs() * ok.abs()).sum(-1, keepdim=True)))
    dv = Pb.transpose(1, 2) @ dOh
    dv_arith = ((PROB + ACC) * Pb + e_P).transpose(1, 2) @ dOh.abs()
    dk = dS.transpose(1, 2) @ qh
    dk_arith = (e_dS + ACC * dS.abs()).transpose(1, 2) @ qh.abs()
    dq = dS @ kh
    dq_arith = (e_dS + ACC * dS.abs()) @ kh.abs()
    out.update(dq=_packed(dq), dq_arith=_packed(dq_arith), dk=_packed(dk), dk_arith=_packed(dk_arith), dv=_packed(dv),
               dv_arith=_packed(dv_arith))
    return out


def attention(q, k, v, cu_q, cu_k, H: int, bias_by_distance=None, o_k=None, lse_k=None, dout=None, mutate=None, drop_last_tile=False):
    """``attention_sample`` over packed samples, concatenated back into packed rows: ``cu_q`` / ``cu_k`` host lists of sample starts
    (self-attention: ``cu_k`` None, the keys are the query rows). ``o_k`` [Mq, 64 H], ``lse_k`` [H, Mq], ``dout`` [Mq, 64 H] as the
    kernels take them. Returns a dict of packed tensors: o, o_arith, dq, dq_arith [Mq, 64 H]; lse, lse_arith [H, Mq]; dk, dk_arith, dv,
    dv_arith [Mk, 64 H] (0 on key rows no sample owns)."""
    cu_k = cu_q if cu_k is None else cu_k
    out = {}
    for b in range(len(cu_q) - 1):
        qs, ks = slice(cu_q[b], cu_q[b + 1]), slice(cu_k[b], cu_k[b + 1])
        r = attention_sample(q[qs], k[ks], v[ks], H, bias_by_distance, None if o_k is None else o_k[qs],
                             None if lse_k is None else lse_k[:, qs], None if dout is None else dout[qs], mutate, drop_last_tile)
        for name, t in r.items():
            if name not in out:
                rows = k.shape[0] if name.startswith(("dk", "dv")) else q.shape[0]
                shape = (H, rows) if name.startswith("lse") else (rows, t.shape[1])
                out[name] = torch.zeros(shape, dtype=torch.float64, device=q.device)
            if name.startswith("lse"):
                out[name][:, qs] = t
            else:
                out[name][ks if name.startswith(("dk", "dv")) else qs] = t
    return out


def attention_error(value, ref: dict, name: str):
    """(|error|, tolerance) of a kernel's bf16 attention output ``name`` (o, dq, dk, dv): half an ulp plus the arithmetic bound; where
    the bound is 0 (no keys, or keys no query sees) the kernel must write exactly 0. ``lse``: fp32 output, the arithmetic bound
    plus an fp32 ulp; -inf where the sample has no keys."""
    v, r, a = value.to(torch.float64), ref[name], ref[name + "_arith"]
    if name == "lse":
        fin = torch.isfinite(r)
        err = torch.where(fin, (v - r).abs(), torch.where(v == r, 0.0, float("inf")))
        return err, torch.where(fin, a + 2 * U * r.abs(), 0.0)
    return (v - r).abs(), torch.where(a > 0, 0.5 * ulp(torch.maximum(v.abs(), r.abs())) + a + FTZ, 0.0)


# ------------------------------------------------------------------------------------------------ sublayer input gradients
def residual_norm_bwd(dy, x, rstd, ln_w, dxn):
    """(dx, arith) of the pre-norm's backward with the residual folded in, from the forward's fp32 ``rstd`` and the bf16 ``dxn``:
    dx = dy + rstd g dxn - x rstd^3 mean(g dxn x). The kernel rounds once to bf16 (within one ulp with its fp32 additions); ``arith``
    bounds its fp32 arithmetic: ROW_EPS times the size of the two terms (the row sum over d in fp32, rstd^3 and the products)."""
    dy, x, dxn = dy.to(torch.float64), x.to(torch.float64), dxn.to(torch.float64)
    r = rstd.to(torch.float64)[:, None]
    g = ln_w.to(torch.float64)
    gd = g * dxn
    d = x.shape[1]
    dx = dy + r * gd - x * r.pow(3) * (gd * x).sum(1, keepdim=True) / d
    arith = ROW_EPS * (r * gd.abs() + x.abs() * r.pow(3) * (gd * x).abs().sum(1, keepdim=True) / d)
    return dx, arith


def dgated(ab, t, t_bound):
    """(d_ab, tolerance without the output's half ulp) in the pair layout, from the kernel's bf16 ``ab`` and t = dy wo in float64 with
    the bound ``t_bound`` of its fp32 accumulation: d_a = t b gelu_new'(a), d_b = t gelu_new(a).

    The kernel rounds t to bf16 first: |bf16(t_kernel) - t| <= e_t = half an ulp + t_bound, which also covers a tie-flip of that
    rounding. d_b = bf16(t bf16(gelu_tanh(a))): gelu within half an ulp plus rel |a| s of gelu_new(a), rel = GELU_TANH_REL (1 + |u|); d_a =
    bf16(bf16(t b) gelu_tanh'(a)): t b within |b| e_t plus half an ulp, gelu' within rel (s + 2 |a ds|) of gelu_new'(a)."""
    a, b = (h.to(torch.float64) for h in split_pairs(ab, dim=1))
    c = math.sqrt(2.0 / math.pi)
    u = c * (a + 0.044715 * a.pow(3))
    rel = GELU_TANH_REL * (1 + u.abs())
    # s = (1 + tanh u) / 2 = sigmoid(2u) and 1 - tanh^2 u = 4 s (1 - s), in forms that keep their relative precision where tanh u is
    # within float64's epsilon of -1 (a below about -6); _t5_ffn_ref's 1 + tanh forms lose it there
    s = torch.sigmoid(2 * u)
    xds = a * 2 * s * torch.sigmoid(-2 * u) * c * (1 + 3 * 0.044715 * a * a)
    g, gp = a * s, s + xds
    xds = xds.abs()
    e_t = 0.5 * ulp(t.abs() + t_bound) + t_bound
    e_g = 0.5 * ulp(g.abs() + rel * a.abs() * s) + rel * a.abs() * s
    e_gp = rel * (s + 2 * xds)
    tb = (t.abs() + e_t) * b.abs()
    tol_b = g.abs() * e_t + (t.abs() + e_t) * e_g
    tol_a = gp.abs() * (b.abs() * e_t + 0.5 * ulp(tb)) + tb * e_gp
    return interleave_pairs(t * b * gp, t * g, dim=1), interleave_pairs(tol_a, tol_b, dim=1)


def bf16_out_error(value, ref, arith, ulps: float = 0.5):
    """(|error|, tolerance) of a bf16 output: ``ulps`` ulp at max(|value|, |ref|) plus the arithmetic bound."""
    v = value.to(torch.float64)
    return (v - ref).abs(), ulps * ulp(torch.maximum(v.abs(), ref.abs())) + arith


def row_blocks(M: int, block: int = BLOCK_ROWS):
    return [slice(r0, min(M, r0 + block)) for r0 in range(0, M, block)]

