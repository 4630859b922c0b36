"""The kernel launches behind each composite C entry point, as the profiler records them: one small call per entry with profiling
on, then the exact sequence of profile tags from the timeline (unprofiled launches -- column-sum finishers, loss finishers, the
unprofiled RMSNorm forward -- leave no tag), and for every gemm_* tag the work the launch reported, 2 M N K. This pins which
kernels each entry runs and in what order, independently of the numbers they compute."""
import pytest
import torch

from thinkdiff_mlre_b200 import _lib as L
from thinkdiff_mlre_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _bf16(*shape, scale=1.0):
    return (torch.randn(*shape, device=DEV) * scale).to(torch.bfloat16)


def _cu(lens):
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    return torch.tensor(cu, dtype=torch.int32, device=DEV)


def _profiled(fn):
    torch.cuda.synchronize()
    L.profile_enable(True)
    try:
        fn()
        torch.cuda.synchronize()
        tags = [t for t, *_ in L.profile_timeline()]
        report = L.profile_report()
    finally:
        L.profile_enable(False)
    return tags, report


def _expect(fn, tags, gemms=None):
    got, report = _profiled(fn)
    assert got == tags
    for tag, (M, N, K) in (gemms or {}).items():
        assert report[tag]["launches"] == 1, tag
        assert report[tag]["work"] == pytest.approx(2.0 * M * N * K, rel=1e-6), tag
    assert {t for t in got if t.startswith("gemm_")} == set(gemms or {})


M, DIN, D = 300, 192, 256


def _aligner():
    torch.manual_seed(0)
    x = _bf16(M, DIN)
    W1, b1 = _bf16(D, DIN, scale=0.05), _bf16(D, scale=0.1)
    W2, b2 = _bf16(D, D, scale=0.05), _bf16(D, scale=0.1)
    g = torch.rand(D, device=DEV) + 0.5
    return x, W1, b1, W2, b2, g


def test_aligner_forward():
    x, W1, b1, W2, b2, g = _aligner()
    _expect(lambda: ops.aligner_fwd(x, W1, b1, W2, b2, g, 1e-6, out_bf16=False, save_for_backward=True),
            ["gemm_fwd1_bias_gelu", "gemm_fwd2_bias_ssq", "rmsnorm_fwd"],
            {"gemm_fwd1_bias_gelu": (M, D, DIN), "gemm_fwd2_bias_ssq": (M, D, D)})


def test_aligner_mse_forward():
    x, W1, b1, W2, b2, g = _aligner()
    target = torch.randn(M, D, device=DEV)
    _expect(lambda: ops.aligner_mse_fwd(x, W1, b1, W2, b2, g, 1e-6, target),
            ["gemm_fwd1_bias_gelu", "gemm_fwd2_bias_ssq", "norm_mse_bwd_fused"],
            {"gemm_fwd1_bias_gelu": (M, D, DIN), "gemm_fwd2_bias_ssq": (M, D, D)})


def test_aligner_backward_all_phases():
    x, W1, b1, W2, b2, g = _aligner()
    _, saved = ops.aligner_fwd(x, W1, b1, W2, b2, g, 1e-6, out_bf16=False, save_for_backward=True)
    bwd = ops.AlignerBackward(x, saved, W2, g, torch.randn(M, D, device=DEV))
    f32 = lambda *s: torch.empty(*s, device=DEV)  # noqa: E731
    dW1, db1, dW2, db2, dg = f32(D, DIN), f32(D), f32(D, D), f32(D), f32(D)
    _expect(lambda: bwd._call(L.BWD_ALL, dW1, db1, dW2, db2, dg),
            ["rmsnorm_bwd", "gemm_dh0_dgelu", "gemm_dW1", "gemm_dW2"],
            {"gemm_dh0_dgelu": (M, D, D), "gemm_dW1": (D, DIN, M), "gemm_dW2": (D, D, M)})


def test_rmsnorm():
    x = _bf16(M, D)
    g = torch.rand(D, device=DEV) + 0.5
    _expect(lambda: ops.rmsnorm_fwd(x, g, out_bf16=True), [])
    _, rstd = ops.rmsnorm_fwd(x, g)
    for want_dg, want_dxsum in ((True, True), (True, False), (False, True), (False, False)):
        _expect(lambda: ops.rmsnorm_bwd(torch.randn(M, D, device=DEV), x, rstd, g, want_dg, want_dxsum), ["rmsnorm_bwd"])


def test_lm_head_and_linear():
    R, K, V = 300, 192, 512
    seq, W = _bf16(R, K), _bf16(V, K, scale=0.05)
    labels = torch.randint(0, V, (R,), device=DEV)
    _expect(lambda: ops.lm_head_ce(seq, W, labels), ["gemm_linear", "masked_ce", "gemm_linear_dx"],
            {"gemm_linear": (R, V, K), "gemm_linear_dx": (R, K, V)})


H, INNER = 2, 128
LENS_Q, LENS_K = [5, 9, 130], [7, 0, 64]


def test_attention_core():
    torch.manual_seed(1)
    cu_q, cu_k = _cu(LENS_Q), _cu(LENS_K)
    Mq, Mk = sum(LENS_Q), sum(LENS_K)
    bias = torch.randn(H, 32, device=DEV)
    q, k, v, do = _bf16(Mq, INNER), _bf16(Mq, INNER), _bf16(Mq, INNER), _bf16(Mq, INNER)
    _expect(lambda: ops.t5_attention_fwd(q, k, v, cu_q, None, max(LENS_Q), max(LENS_Q), H, bias), ["attn_fwd"])
    o, lse = ops.t5_attention_fwd(q, k, v, cu_q, None, max(LENS_Q), max(LENS_Q), H, bias)
    _expect(lambda: ops.t5_attention_bwd(do, q, k, v, o, lse, cu_q, None, max(LENS_Q), max(LENS_Q), H, bias),
            ["attn_bwd_delta", "attn_bwd_dkdv", "attn_bwd_dq"])
    kc, vc = _bf16(Mk, INNER), _bf16(Mk, INNER)
    _expect(lambda: ops.t5_attention_fwd(q, kc, vc, cu_q, cu_k, max(LENS_Q), max(LENS_K), H), ["attn_fwd"])
    o, lse = ops.t5_attention_fwd(q, kc, vc, cu_q, cu_k, max(LENS_Q), max(LENS_K), H)
    _expect(lambda: ops.t5_attention_bwd(do, q, kc, vc, o, lse, cu_q, cu_k, max(LENS_Q), max(LENS_K), H),
            ["attn_bwd_delta", "attn_bwd_dkdv", "attn_bwd_dq"])


def test_ffn():
    torch.manual_seed(2)
    d, d_ff = 128, 256
    x, wi, wo = _bf16(M, d), _bf16(2 * d_ff, d, scale=0.05), _bf16(d, d_ff, scale=0.05)
    ln_w = torch.rand(d, device=DEV) + 0.5
    _expect(lambda: ops.t5_ffn_fwd(x, wi, wo, ln_w, 1e-6), ["ffn_norm", "gemm_ffn_gate", "gemm_ffn_out"],
            {"gemm_ffn_gate": (M, 2 * d_ff, d), "gemm_ffn_out": (M, d, d_ff)})
    _, rstd, ab, _ = ops.t5_ffn_fwd(x, wi, wo, ln_w, 1e-6)
    _expect(lambda: ops.t5_ffn_bwd(_bf16(M, d), x, rstd, ab, wi, wo, ln_w), ["gemm_ffn_dgate", "gemm_ffn_dx", "ffn_norm_bwd"],
            {"gemm_ffn_dgate": (M, d_ff, d), "gemm_ffn_dx": (M, d, 2 * d_ff)})


def test_attention_sublayers():
    torch.manual_seed(3)
    d = 128
    cu_q, cu_k = _cu(LENS_Q), _cu(LENS_K)
    Mq, Mk = sum(LENS_Q), sum(LENS_K)
    x, enc, dy = _bf16(Mq, d), _bf16(Mk, d), _bf16(Mq, d)
    ln_w = torch.rand(d, device=DEV) + 0.5
    w_qkv, w_q, w_kv = (_bf16(n, d, scale=0.05) for n in (3 * INNER, INNER, 2 * INNER))
    wo = _bf16(d, INNER, scale=0.05)
    bias = torch.randn(H, 32, device=DEV)
    lq, lk = max(LENS_Q), max(LENS_K)

    _expect(lambda: ops.t5_self_attention_layer_fwd(x, w_qkv, wo, ln_w, 1e-6, bias, cu_q, lq, H),
            ["sa_norm", "gemm_sa_qkv", "attn_fwd", "gemm_sa_out"],
            {"gemm_sa_qkv": (Mq, 3 * INNER, d), "gemm_sa_out": (Mq, d, INNER)})
    _, rstd, qkv, o, lse = ops.t5_self_attention_layer_fwd(x, w_qkv, wo, ln_w, 1e-6, bias, cu_q, lq, H)
    _expect(lambda: ops.t5_self_attention_layer_bwd(dy, x, rstd, qkv, o, lse, w_qkv, wo, ln_w, bias, cu_q, lq, H),
            ["gemm_sa_do", "attn_bwd_delta", "attn_bwd_dkdv", "attn_bwd_dq", "gemm_sa_dx", "sa_norm_bwd"],
            {"gemm_sa_do": (Mq, INNER, d), "gemm_sa_dx": (Mq, d, 3 * INNER)})

    _expect(lambda: ops.t5_cross_attention_layer_fwd(x, enc, w_q, w_kv, wo, ln_w, 1e-6, cu_q, cu_k, lq, lk, H),
            ["ca_norm", "gemm_ca_q", "gemm_ca_kv", "attn_fwd", "gemm_ca_out"],
            {"gemm_ca_q": (Mq, INNER, d), "gemm_ca_kv": (Mk, 2 * INNER, d), "gemm_ca_out": (Mq, d, INNER)})
    _, rstd, q, kv, o, lse = ops.t5_cross_attention_layer_fwd(x, enc, w_q, w_kv, wo, ln_w, 1e-6, cu_q, cu_k, lq, lk, H)
    _expect(lambda: ops.t5_cross_attention_layer_bwd(dy, x, rstd, q, kv, o, lse, w_q, w_kv, wo, ln_w, cu_q, cu_k, lq, lk, H),
            ["gemm_ca_do", "attn_bwd_delta", "attn_bwd_dkdv", "attn_bwd_dq", "gemm_ca_dq", "gemm_ca_denc", "ca_norm_bwd"],
            {"gemm_ca_do": (Mq, INNER, d), "gemm_ca_dq": (Mq, d, INNER), "gemm_ca_denc": (Mk, d, 2 * INNER)})


def test_pack():
    flat, flat2 = _bf16(40, 64), _bf16(30, 64)
    cu = _cu([5, 9, 0, 3])
    starts = torch.tensor([0, 10, 20, 30], dtype=torch.int64, device=DEV)
    _expect(lambda: ops.pack_varlen(flat, starts, cu, 17, want_index=True), ["pack_varlen"])
    starts2 = torch.tensor([0, -1, 20, -11], dtype=torch.int64, device=DEV)
    _expect(lambda: ops.pack_varlen2(flat, flat2, starts2, cu, 17), ["pack_varlen"])
    _expect(lambda: ops.pack_padded(flat, starts, cu, 9), ["pack_padded"])
