#!/usr/bin/env python
"""Timing of the T5 decoder's gated-GELU feed-forward sublayer on packed rows (T5LayerFF; td_t5_ffn_fwd / _bwd) on one B200,
forward and forward + backward (input gradient only, frozen weights), next to two references on the same GPU and inputs: eager
transformers T5LayerFF (bf16 weights, bf16 autocast, dropout off) with autograd, and a cuBLAS floor -- the three torch.matmul calls
of each direction alone (xn wi_0^T, xn wi_1^T, g wo^T; dy wo, d_a wi_0, d_b wi_1), with no norm, gate or residual work at all.

Shapes: Flan-T5-XXL, d = 4096, d_ff = 10240. M = the decoder row counts of cfg2 and cfg5 drawn as scripts/bench_t5_attention.py
draws them (64 and 128 sequences of U{8..128} rows from the same seeded generator), and M = 8192. FLOPs: 6 M d d_ff per direction
(the three GEMMs). The frozen weights alone are 252 MB, twice the 126 MB L2, so every call streams them from HBM; activations stay
in L2 where they fit. One JSON line on stdout.

    python scripts/bench_t5_ffn.py > profiles/rNN_t5_ffn.json
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib as L

D, D_FF, EPS = 4096, 10240, 1e-6
PEAK_FLOPS = 2250e12  # B200 data sheet, dense bf16 (1000 W card)
REPS = 20


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        smi = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        smi = None
    return {"torch_name": name, "nvidia_smi": smi}


def timed(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / REPS


def decoder_rows():
    """Row counts of the cfg2 / cfg5 decoder batches, from the generator sequence of bench_t5_attention.py (seed 0: cfg2's 64 query
    then 64 key lengths, then cfg5's 128 query lengths)."""
    gen = torch.Generator().manual_seed(0)
    cfg2 = torch.randint(8, 129, (64,), generator=gen)
    torch.randint(1, 257, (64,), generator=gen)
    cfg5 = torch.randint(8, 129, (128,), generator=gen)
    return {"cfg2": int(cfg2.sum()), "cfg5": int(cfg5.sum()), "m8192": 8192}


def hf_layer(wi_0, wi_1, wo, ln_w):
    import transformers
    from transformers.models.t5.modeling_t5 import T5LayerFF

    cfg = transformers.T5Config(d_model=D, d_ff=D_FF, feed_forward_proj="gated-gelu", dropout_rate=0.0)
    with torch.device("cuda"):
        layer = T5LayerFF(cfg).eval()
    with torch.no_grad():
        layer.DenseReluDense.wi_0.weight.copy_(wi_0)
        layer.DenseReluDense.wi_1.weight.copy_(wi_1)
        layer.DenseReluDense.wo.weight.copy_(wo)
        layer.layer_norm.weight.copy_(ln_w)
    return layer.to(torch.bfloat16).requires_grad_(False)


def run_shape(M, w, layer, raw):
    wi_0, wi_1, wo = raw
    g = torch.Generator(device="cuda").manual_seed(M)
    x = torch.randn((M, D), generator=g, device="cuda").to(torch.bfloat16)
    dy = torch.randn((M, D), generator=g, device="cuda").to(torch.bfloat16)

    def ours_fwd():
        return td.ops.t5_ffn_fwd(x, w.wi, w.wo, w.ln_weight, EPS, want_ab=False)[0]

    def ours_fwd_bwd():
        out, rstd, ab, _ = td.ops.t5_ffn_fwd(x, w.wi, w.wo, w.ln_weight, EPS)
        return td.ops.t5_ffn_bwd(dy, x, rstd, ab, w.wi, w.wo, w.ln_weight)[0]

    def hf_fwd():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return layer(x)

    def hf_fwd_bwd():
        xh = x.detach().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = layer(xh)
        out.backward(dy)
        return xh.grad

    a = torch.randn((M, D_FF), generator=g, device="cuda").to(torch.bfloat16)
    b = torch.randn((M, D_FF), generator=g, device="cuda").to(torch.bfloat16)

    def floor_fwd():
        torch.matmul(x, wi_0.t())
        torch.matmul(x, wi_1.t())
        torch.matmul(a, wo.t())

    def floor_bwd():
        torch.matmul(dy, wo)
        torch.matmul(a, wi_0)
        torch.matmul(b, wi_1)

    flops = 6.0 * M * D * D_FF
    res = {"M": M, "flops_per_direction": flops}
    res["fwd_ms"] = timed(ours_fwd)
    res["fwd_bwd_ms"] = timed(ours_fwd_bwd)
    res["eager_hf_fwd_ms"] = timed(hf_fwd)
    res["eager_hf_fwd_bwd_ms"] = timed(hf_fwd_bwd)
    res["cublas_floor_fwd_ms"] = timed(floor_fwd)
    res["cublas_floor_fwd_bwd_ms"] = res["cublas_floor_fwd_ms"] + timed(floor_bwd)
    for key, fl in (("fwd", flops), ("fwd_bwd", 2 * flops)):
        res[key + "_tflops"] = fl / res[key + "_ms"] / 1e9
        res[key + "_share_of_datasheet_bf16"] = fl / PEAK_FLOPS * 1e3 / res[key + "_ms"]
        res["eager_hf_" + key + "_tflops"] = fl / res["eager_hf_" + key + "_ms"] / 1e9
        res["cublas_floor_" + key + "_tflops"] = fl / res["cublas_floor_" + key + "_ms"] / 1e9
        res["speedup_" + key + "_vs_eager_hf"] = res["eager_hf_" + key + "_ms"] / res[key + "_ms"]
        res["ratio_" + key + "_to_cublas_floor"] = res[key + "_ms"] / res["cublas_floor_" + key + "_ms"]
    L.profile_enable(True)
    for _ in range(REPS):
        ours_fwd_bwd()
    torch.cuda.synchronize()
    prof = L.profile_report()
    L.profile_enable(False)
    res["kernels"] = {t: {"ms_per_launch": r["ms"] / r["launches"], "work_per_launch": r["work"] / r["launches"],
                          "tflops": (r["work"] / r["ms"] / 1e9) if t.startswith("gemm") else None} for t, r in prof.items()}
    with torch.no_grad():
        o, h = ours_fwd().float(), hf_fwd().float()
    res["rel_diff_out_vs_eager_hf"] = float((o - h).norm() / h.norm())
    print(M, json.dumps(res), file=sys.stderr)
    return res


def main():
    assert torch.cuda.is_available(), "bench_t5_ffn.py measures on the GPU; there is no CPU path"
    g = torch.Generator(device="cuda").manual_seed(0)
    wi_0 = (torch.randn((D_FF, D), generator=g, device="cuda") * D ** -0.5).to(torch.bfloat16)
    wi_1 = (torch.randn((D_FF, D), generator=g, device="cuda") * D ** -0.5).to(torch.bfloat16)
    wo = (torch.randn((D, D_FF), generator=g, device="cuda") * D_FF ** -0.5).to(torch.bfloat16)
    ln_w = (1.0 + 0.1 * torch.randn((D,), generator=g, device="cuda")).to(torch.bfloat16).float()
    w = td.T5FeedForwardWeights(wi_0, wi_1, wo, ln_w, EPS)
    layer = hf_layer(wi_0, wi_1, wo, ln_w)
    out = {"card": card(), "d_model": D, "d_ff": D_FF, "reps": REPS,
           "note": "times from CUDA events over REPS back-to-back calls after 3 warm-up calls; the 252 MB of frozen weights exceed "
                   "the 126 MB L2, activations stay in L2 where they fit; per-kernel times come from a separate profiled pass "
                   "(td_profile_enable: events between launches, so they include each kernel's prologue); the cuBLAS floor is the "
                   "three matmuls of each direction alone"}
    for name, M in decoder_rows().items():
        out[name] = run_shape(M, w, layer, (wi_0, wi_1, wo))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
