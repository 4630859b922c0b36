"""GPU parity of the T5 gated-GELU FFN sublayer (td_t5_ffn_fwd / _bwd: the gated, gated-backward and residual GEMM epilogues of
csrc/gemm_sm100.cuh and the residual norm backward of csrc/rowops_sm100.cuh) through the C ABI and the autograd boundary: each stage
against a reference on the kernel's own inputs (ab, gated, d_ab), the sublayer's out and dx against the float64 reference on the
same bf16 inputs, the sublayer against transformers' T5LayerFF under bf16 autocast, determinism, the inference path, M = 0, the
rejected arguments, and a frozen_linear -> t5_layer_ff chain under autograd. M crosses the 128- and 256-row tile edges and makes
stream-K tails appear and disappear; (512, 1056) has a partial last n-tile in every GEMM that runs over d_ff."""
import pytest
import torch

import _t5_ffn_ref as ref
import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib, ops
from thinkdiff_mlre_b200.t5 import T5FeedForwardWeights

pytestmark = pytest.mark.gpu

MS = [1, 127, 128, 129, 255, 256, 257, 1000, 4352]
DIMS = [(512, 1024), (512, 1056), (4096, 10240)]
EPS = 1e-6
_weights = {}


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _ulp(t, floor=2.0 ** -14):
    """bf16 ulp at |t| (float64), taken at |t| >= floor: below that the bf16 spacing is finer than the fp32 accumulation error."""
    e = torch.floor(torch.log2(t.double().abs().clamp_min(floor)))
    return torch.pow(2.0, e - 7)


def _raw(d, d_ff):
    """Seeded bf16 weights (wi_0, wi_1, wo) and an fp32 norm weight with bf16 values, on the GPU; cached per shape."""
    if (d, d_ff) not in _weights:
        g = torch.Generator(device="cuda").manual_seed(d * 7 + d_ff)
        wi_0 = (torch.randn((d_ff, d), generator=g, device="cuda") * d ** -0.5).to(torch.bfloat16)
        wi_1 = (torch.randn((d_ff, d), generator=g, device="cuda") * d ** -0.5).to(torch.bfloat16)
        wo = (torch.randn((d, d_ff), generator=g, device="cuda") * d_ff ** -0.5).to(torch.bfloat16)
        ln_w = (1.0 + 0.1 * torch.randn((d,), generator=g, device="cuda")).to(torch.bfloat16).float()
        _weights[(d, d_ff)] = (wi_0, wi_1, wo, ln_w, T5FeedForwardWeights(wi_0, wi_1, wo, ln_w, EPS))
    return _weights[(d, d_ff)]


def _inputs(M, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((M, d), generator=g, device="cuda").to(torch.bfloat16)
    dy = torch.randn((M, d), generator=g, device="cuda").to(torch.bfloat16)
    return x, dy


@pytest.mark.parametrize("dims", DIMS, ids=lambda t: f"d{t[0]}_ff{t[1]}")
@pytest.mark.parametrize("M", MS)
def test_ffn_stages_and_sublayer_against_references(M, dims):
    d, d_ff = dims
    wi_0, wi_1, wo, ln_w, w = _raw(d, d_ff)
    x, dy = _inputs(M, d, seed=M + d_ff)
    out, rstd, ab, gated = ops.t5_ffn_fwd(x, w.wi, w.wo, w.ln_weight, EPS, want_ab=True, want_gated=True)
    dx, d_ab = ops.t5_ffn_bwd(dy, x, rstd, ab, w.wi, w.wo, w.ln_weight, want_d_ab=True)
    torch.cuda.synchronize()

    # 1. ab = xn . wi^T (interleaved), xn from the same norm kernel
    xn, rstd_n = ops.rmsnorm_fwd(x, ln_w, EPS, out_bf16=True)
    assert torch.equal(rstd, rstd_n)
    a, b = T5FeedForwardWeights.split(ab, dim=1)
    for got, wt in ((a, wi_0), (b, wi_1)):
        want = xn.double() @ wt.double().t()
        assert _rel(got, want) <= 2e-3
        # near zero the tensor core's fp32 sum over d terms of size ~1/sqrt(d) errs by ~1e-6, more than a bf16 ulp there
        assert bool(((got.double() - want).abs() <= 2 * _ulp(want, floor=2.0 ** -10)).all())

    # 2. gated from the kernel's own a, b: >= 99 % bit-equal, and every element within 1 bf16 ulp of the oracle -- evaluated with
    # gelu_new(a) nudged by 4e-6 either way, since where gelu_new(a) lies that close to a bf16 tie the kernel's fp32 value may round
    # it to the other neighbour, and the product then moves by up to two ulps
    g_ref = ref.gated_staged(a, b)
    near = torch.minimum(*((gated.double() - ref.gated_staged(a, b, nudge=f)).abs() for f in (1 - 4e-6, 1 + 4e-6)))
    assert bool((near <= _ulp(g_ref)).all())
    assert float((gated == g_ref).float().mean()) >= 0.99

    # 3. d_ab from the kernel's own ab, t = dy . wo in float64
    d_a_ref, d_b_ref = ref.dgated_staged(dy.double() @ wo.double(), a, b)
    d_a, d_b = T5FeedForwardWeights.split(d_ab, dim=1)
    assert _rel(d_a, d_a_ref) <= 5e-3 and _rel(d_b, d_b_ref) <= 5e-3

    # 4. the sublayer against the float64 reference on the same bf16 inputs
    r_out, r_dx = ref.layer_ff_with_grad(x, ln_w, wi_0, wi_1, wo, EPS, dy)
    assert _rel(out, r_out) <= 5e-3
    assert _rel(dx, r_dx) <= 1e-2


@pytest.mark.parametrize("M,dims", [(1000, (512, 1024)), (257, (512, 1056)), (4352, (4096, 10240))])
def test_sublayer_is_closer_to_fp32_than_hf_under_autocast(M, dims):
    transformers = pytest.importorskip("transformers")
    from transformers.models.t5.modeling_t5 import T5LayerFF

    d, d_ff = dims
    wi_0, wi_1, wo, ln_w, w = _raw(d, d_ff)
    x, dy = _inputs(M, d, seed=3 * M)
    cfg = transformers.T5Config(d_model=d, d_ff=d_ff, feed_forward_proj="gated-gelu", dropout_rate=0.0)
    layer = T5LayerFF(cfg).eval()
    with torch.no_grad():
        layer.DenseReluDense.wi_0.weight.copy_(wi_0.float().cpu())
        layer.DenseReluDense.wi_1.weight.copy_(wi_1.float().cpu())
        layer.DenseReluDense.wo.weight.copy_(wo.float().cpu())
        layer.layer_norm.weight.copy_(ln_w.cpu())
    layer = layer.to(device="cuda", dtype=torch.bfloat16).requires_grad_(False)
    xh = x.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out_hf = layer(xh)
    out_hf.backward(dy)
    xk = x.clone().requires_grad_(True)
    out_k = td.t5_layer_ff(xk, T5FeedForwardWeights.from_module(layer).to("cuda"))
    out_k.backward(dy)
    r_out, r_dx = ref.layer_ff_with_grad(x, ln_w, wi_0, wi_1, wo, EPS, dy)
    assert _rel(out_k, r_out) <= 1.25 * _rel(out_hf, r_out)
    assert _rel(xk.grad, r_dx) <= 1.25 * _rel(xh.grad, r_dx)


def test_bit_identical_across_runs_and_inference_path_matches():
    d, d_ff = 4096, 10240
    _, _, _, _, w = _raw(d, d_ff)
    x, dy = _inputs(4352, d, seed=11)
    runs = []
    for _ in range(2):
        out, rstd, ab, _ = ops.t5_ffn_fwd(x, w.wi, w.wo, w.ln_weight, EPS)
        dx, d_ab = ops.t5_ffn_bwd(dy, x, rstd, ab, w.wi, w.wo, w.ln_weight, want_d_ab=True)
        runs.append((out, rstd, ab, dx, d_ab))
    for t0, t1 in zip(*runs):
        assert torch.equal(t0, t1)
    out_inf, rstd_inf, ab_inf, _ = ops.t5_ffn_fwd(x, w.wi, w.wo, w.ln_weight, EPS, want_ab=False)
    assert ab_inf is None and torch.equal(out_inf, runs[0][0]) and torch.equal(rstd_inf, runs[0][1])
    with torch.no_grad():  # the autograd boundary takes the inference path when no gradient is needed
        assert torch.equal(td.t5_layer_ff(x, w), runs[0][0])


def test_empty_batch_is_a_no_op():
    _, _, _, _, w = _raw(512, 1024)
    x = torch.empty((0, 512), dtype=torch.bfloat16, device="cuda")
    out, rstd, ab, _ = ops.t5_ffn_fwd(x, w.wi, w.wo, w.ln_weight, EPS)
    dx, _ = ops.t5_ffn_bwd(x, x, rstd, ab, w.wi, w.wo, w.ln_weight)
    assert out.shape == (0, 512) and ab.shape == (0, 2048) and dx.shape == (0, 512)
    lib = _lib.lib()
    assert lib.td_t5_ffn_fwd(None, 0, 512, 1024, None, EPS, None, None, None, None, None, None, None, 0, None) == 0
    assert lib.td_t5_ffn_bwd(None, None, None, None, None, None, None, 0, 512, 1024, None, None, None, 0, None) == 0


def test_rejected_arguments():
    lib = _lib.lib()
    _, _, _, _, w = _raw(512, 1024)
    M, d, d_ff = 64, 512, 1024
    x, _ = _inputs(M, d, seed=5)
    out = torch.empty_like(x)
    rstd = torch.empty((M,), dtype=torch.float32, device="cuda")
    ws_bytes = lib.td_t5_ffn_workspace_bytes(M, d, d_ff)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    P = _lib.ptr

    def fwd(x_, d_=d, d_ff_=d_ff, wi=w.wi, ws_bytes_=ws_bytes):
        return lib.td_t5_ffn_fwd(P(x_), M, d_, d_ff_, P(w.ln_weight), EPS, P(wi), P(w.wo), P(out), P(rstd), None, None, P(ws), ws_bytes_,
                                 _lib.stream_ptr())

    assert fwd(x) == 0
    assert fwd(x, d_ff_=1000) != 0 and "d_ff" in _lib.last_error()  # d_ff % 32
    assert fwd(x, d_=480) != 0 and "d %" in _lib.last_error()        # d % 64
    assert fwd(x, ws_bytes_=ws_bytes - 256) != 0 and "workspace" in _lib.last_error()
    buf = torch.empty((M * d + 8,), dtype=torch.bfloat16, device="cuda")
    assert fwd(buf[1 : 1 + M * d].view(M, d)) != 0 and "aligned" in _lib.last_error()
    wi_bad = torch.empty((2 * d_ff * d + 8,), dtype=torch.bfloat16, device="cuda")[4 : 4 + 2 * d_ff * d]
    assert fwd(x, wi=wi_bad) != 0 and "aligned" in _lib.last_error()
    dx = torch.empty_like(x)
    assert lib.td_t5_ffn_bwd(P(x), P(x), P(rstd), P(w.ln_weight), None, P(w.wi), P(w.wo), M, d, d_ff, P(dx), None, P(ws), ws_bytes,
                             _lib.stream_ptr()) != 0  # the backward needs the forward's ab
    with pytest.raises(TypeError):
        ops.t5_ffn_bwd(x, x, rstd, None, w.wi, w.wo, w.ln_weight)
    wi_0 = torch.zeros((d_ff, d), device="cuda", requires_grad=True)
    with pytest.raises(NotImplementedError, match="require grad"):
        T5FeedForwardWeights(wi_0, wi_0.detach(), torch.zeros((d, d_ff), device="cuda"), torch.ones(d, device="cuda"))


def test_frozen_linear_then_ffn_under_autograd_matches_the_reference_chain():
    d, d_ff, d_in, M = 4096, 10240, 1024, 1000
    wi_0, wi_1, wo, ln_w, w = _raw(d, d_ff)
    g = torch.Generator(device="cuda").manual_seed(17)
    W = (torch.randn((d, d_in), generator=g, device="cuda") * d_in ** -0.5).to(torch.bfloat16)
    x0 = torch.randn((M, d_in), generator=g, device="cuda").to(torch.bfloat16).requires_grad_(True)
    dy = torch.randn((M, d), generator=g, device="cuda").to(torch.bfloat16)
    out = td.t5_layer_ff(td.frozen_linear(x0, W), w)
    out.backward(dy)
    xr = x0.detach().double().requires_grad_(True)
    ref.layer_ff(xr @ W.double().t(), *(t.double() for t in (ln_w, wi_0, wi_1, wo)), EPS).backward(dy.double())
    assert x0.grad.dtype == torch.bfloat16
    assert _rel(x0.grad, xr.grad) <= 1e-2
