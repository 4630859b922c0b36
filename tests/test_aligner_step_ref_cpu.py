"""CPU: the float64 staged reference of the fused train step (tests/_aligner_step_ref.py, which the production-width GPU parity
test compares the kernels with) restates the closed-form oracle's rounding points exactly."""
import torch

import _aligner_step_ref as R
from oracle import aligner_ref


def test_ulp_is_the_bf16_spacing():
    v = torch.tensor([1.0, 1.5, 0.75, -3.0, 2.0 ** -126, 0.0], dtype=torch.float64)
    want = torch.tensor([2.0 ** -7, 2.0 ** -7, 2.0 ** -8, 2.0 ** -6, 2.0 ** -133, 2.0 ** -133], dtype=torch.float64)
    assert torch.equal(R.ulp(v), want)
    # a bf16 value and its neighbour are one ulp apart
    b = torch.tensor([1.0, 3.0, -0.1], dtype=torch.bfloat16)
    up = (b.view(torch.int16) + 1).view(torch.bfloat16).double()
    assert torch.equal((up - b.double()).abs(), R.ulp(b.double()))


def test_staged_reference_matches_closed_form_oracle():
    M, din, d = 37, 128, 256
    params = aligner_ref.init_params_numpy(din, d, seed=3)
    gen = torch.Generator().manual_seed(0)
    x = torch.randn((M, din), generator=gen).to(torch.bfloat16)
    t = torch.randn((M, d), generator=gen).to(torch.bfloat16)
    W1, b1, W2, b2 = (params[k].to(torch.bfloat16) for k in ("0.weight", "0.bias", "2.weight", "2.bias"))
    g = params["3.weight"]

    fwd = aligner_ref.aligner_fwd_bwd_manual(x.float(), params, regime="bf16")
    dy = 2.0 * (fwd["y"] - t.float()) / (M * d)
    out = aligner_ref.aligner_fwd_bwd_manual(x.float(), params, dy=dy, regime="bf16")

    # forward: every stage from the previous stage's (here: the reference's own) bf16 output, bit-identical to the oracle
    acc, _ = R.product(x, W1, b1)
    h0 = R.bf16(acc)
    assert torch.equal(h0, out["h0"].double())
    h1 = R.bf16(R.gelu64(h0))
    assert torch.equal(h1, out["h1"].double())
    acc, _ = R.product(h1, W2, b2)
    h2 = R.bf16(acc)
    assert torch.equal(h2, out["h2"].double())

    # norm + MSE + norm backward (the oracle keeps y in fp32 before forming dy; the reference does not round it)
    n = R.norm_mse(h2, g, t, aligner_ref.EPS, 2.0 / (M * d))
    torch.testing.assert_close(n["rstd"], out["rstd"].double(), rtol=2e-7, atol=0)
    torch.testing.assert_close(n["y"], out["y"].double(), rtol=2e-7, atol=1e-12)
    dh2 = R.bf16(n["dh2"])
    off = (dh2 - out["dh2"].double()).abs()
    assert bool((off <= R.ulp(out["dh2"].double())).all()) and float((off == 0).double().mean()) >= 0.99
    torch.testing.assert_close((n["dy"] * n["xhat"]).sum(0), out["dg"].double(), rtol=1e-5, atol=1e-9)

    # backward stages from the oracle's dh2
    dh2 = out["dh2"].double()
    acc, bound = R.product(dh2, W2.T)  # dh1 = dh2 W2
    dh0 = R.bf16(R.bf16(acc) * R.gelu_grad64(h0))
    assert torch.equal(dh0, out["dh0"].double())
    err, tol = R.gemm_error("dgelu", dh0, acc, bound, R.gelu_grad64(h0))
    assert bool((err <= tol).all())
    for name, (a, b) in {"dW2": (dh2, h1), "dW1": (dh0, x)}.items():
        acc, bound = R.contract_rows(a, b)
        torch.testing.assert_close(acc, out[name].double(), rtol=1e-6, atol=0, msg=name)
        err, tol = R.gemm_error("f32", out[name], acc, bound)
        assert bool((err <= tol).all()), name
    torch.testing.assert_close(dh2.sum(0), out["db2"].double(), rtol=1e-6, atol=0)
    torch.testing.assert_close(dh0.sum(0), out["db1"].double(), rtol=1e-6, atol=0)


def test_gemm_error_rejects_a_one_ulp_shift_of_a_bf16_output():
    gen = torch.Generator().manual_seed(1)
    a = torch.randn((64, 512), generator=gen).to(torch.bfloat16)
    b = torch.randn((96, 512), generator=gen).to(torch.bfloat16)
    acc, bound = R.product(a, b)
    h = R.bf16(acc)
    err, tol = R.gemm_error("bf16", h, acc, bound)
    assert bool((err <= tol).all())
    up = (h.to(torch.bfloat16).view(torch.int16) + 1).view(torch.bfloat16)
    err, tol = R.gemm_error("bf16", up, acc, bound)
    assert float((err > tol).double().mean()) > 0.9
