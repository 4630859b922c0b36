#!/usr/bin/env python
"""Timing of the frozen T5 decoder block on packed rows (t5_decoder_block: td_t5_self_attention_layer_*, td_t5_cross_attention_layer_*,
td_t5_ffn_*) on one B200, forward (inference) and forward + backward (gradients into the decoder rows and the fp32 aligner rows), next
to eager transformers T5Block (bf16 weights, bf16 autocast, dropout off) with autograd on the zero-padded batch + masks, on the same
GPU and inputs; then the 24-block stack (t5_decoder_stack) forward + backward at cfg2.

Shapes: Flan-T5-XXL, d = 4096, 64 heads of d_kv 64, d_ff = 10240. Decoder and aligner lengths are drawn with the generator sequence
of scripts/bench_t5_attention.py (seed 0: cfg2 64 decoder lengths U{8..128} then 64 aligner lengths U{1..256}, cfg5 128 of
U{8..128} then 128 of U{1..1024}). Weights are seeded; q / k rows are scaled so the attention scores stay O(1), and in the stack the
o / wo projections by 1/sqrt(72) more, so that the residual stream stays O(1) over 72 sublayers. FLOPs are computed from shapes:
2 M N K per GEMM plus the visible (query, key) pairs of the attention (4 x 64 H per pair forward, 10 x 64 H backward). One JSON
line on stdout.

    python scripts/bench_t5_decoder_block.py > profiles/rNN_t5_decoder_block.json
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib as L

D, H, D_FF, EPS, N_BLOCKS = 4096, 64, 10240, 1e-6, 24
INNER = 64 * H
PEAK_FLOPS = 2250e12  # B200 data sheet, dense bf16 (1000 W card)
REPS = 10
NEG = torch.finfo(torch.float32).min


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        smi = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        smi = None
    return {"torch_name": name, "nvidia_smi": smi}


def timed(fn, reps=REPS):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def shapes():
    gen = torch.Generator().manual_seed(0)
    out = {}
    for name, B, l_hi in (("cfg2", 64, 256), ("cfg5", 128, 1024)):
        lens_q = torch.randint(8, 129, (B,), generator=gen).tolist()
        lens_k = torch.randint(1, l_hi + 1, (B,), generator=gen).tolist()
        out[name] = (lens_q, lens_k)
    return out


def raw_block(g, o_scale=1.0):
    """Seeded bf16 weights of one block in T5Block state-dict naming (fp32 norm weights with bf16 values)."""
    def lin(n_out, n_in, s=1.0):
        return (torch.randn((n_out, n_in), generator=g, device="cuda") * s * n_in ** -0.5).to(torch.bfloat16)

    def ln():
        return (1.0 + 0.1 * torch.randn((D,), generator=g, device="cuda")).to(torch.bfloat16).float()

    sd = {}
    for i, a in ((0, "SelfAttention"), (1, "EncDecAttention")):
        p = f"layer.{i}.{a}."
        sd[p + "q.weight"], sd[p + "k.weight"], sd[p + "v.weight"] = lin(INNER, D, 0.25), lin(INNER, D, 0.25), lin(INNER, D)
        sd[p + "o.weight"] = lin(D, INNER, o_scale)
        sd[f"layer.{i}.layer_norm.weight"] = ln()
    f = "layer.2.DenseReluDense."
    sd[f + "wi_0.weight"], sd[f + "wi_1.weight"], sd[f + "wo.weight"] = lin(D_FF, D), lin(D_FF, D), lin(D, D_FF, o_scale)
    sd["layer.2.layer_norm.weight"] = ln()
    return sd


def flops(lens_q, lens_k):
    Mq, Mk = sum(lens_q), sum(lens_k)
    self_pairs = sum(t * (t + 1) // 2 for t in lens_q)
    cross_pairs = sum(t * n for t, n in zip(lens_q, lens_k))
    gemm_f = 2.0 * Mq * D * (3 * INNER + INNER) + 2.0 * Mq * D * (2 * INNER) + 2.0 * Mk * D * 2 * INNER + 6.0 * Mq * D * D_FF
    gemm_b = 2.0 * Mq * D * (INNER + 3 * INNER) + 2.0 * Mq * D * (2 * INNER) + 2.0 * Mk * D * 2 * INNER + 6.0 * Mq * D * D_FF
    attn_f, attn_b = 4.0 * 64 * H * (self_pairs + cross_pairs), 10.0 * 64 * H * (self_pairs + cross_pairs)
    return {"rows_q": Mq, "rows_k": Mk, "self_pairs": self_pairs, "cross_pairs": cross_pairs, "fwd": gemm_f + attn_f,
            "fwd_bwd": gemm_f + attn_f + gemm_b + attn_b, "gemm_share_fwd": gemm_f / (gemm_f + attn_f)}


def cu(lens):
    return torch.tensor([0] + torch.tensor(lens).cumsum(0).tolist(), dtype=torch.int32, device="cuda")


def pad(x, lens, L):
    out = x.new_zeros((len(lens), L, x.shape[1]))
    r = 0
    for b, n in enumerate(lens):
        out[b, :n] = x[r : r + n]
        r += n
    return out


def hf_block(sd, table):
    import transformers
    from transformers.models.t5.modeling_t5 import T5Block

    cfg = transformers.T5Config(d_model=D, d_kv=64, d_ff=D_FF, num_heads=H, feed_forward_proj="gated-gelu", dropout_rate=0.0, is_decoder=True,
                                use_cache=False, relative_attention_num_buckets=32, relative_attention_max_distance=128)
    with torch.device("cuda"):
        blk = T5Block(cfg, has_relative_attention_bias=True, layer_idx=0).eval()
    full = dict(sd)
    full["layer.0.SelfAttention.relative_attention_bias.weight"] = table
    blk.load_state_dict({k: v.float() for k, v in full.items()})
    return blk.to(torch.bfloat16).requires_grad_(False)


def run_block(name, lens_q, lens_k, w, bias, blk):
    cuq, cuk = cu(lens_q), cu(lens_k)
    T, Lk = max(lens_q), max(lens_k)
    g = torch.Generator(device="cuda").manual_seed(len(lens_q))
    x = torch.randn((sum(lens_q), D), generator=g, device="cuda").to(torch.bfloat16)
    enc = torch.randn((sum(lens_k), D), generator=g, device="cuda").to(torch.bfloat16).float()
    dy = torch.randn((sum(lens_q), D), generator=g, device="cuda").to(torch.bfloat16)

    def ours_fwd():
        with torch.no_grad():
            return td.t5_decoder_block(x, enc, cuq, cuk, T, Lk, w, bias)

    def ours_fwd_bwd():
        xk, ek = x.detach().requires_grad_(True), enc.detach().requires_grad_(True)
        td.t5_decoder_block(xk, ek, cuq, cuk, T, Lk, w, bias).backward(dy)
        return ek.grad

    xp, ep, dyp = pad(x, lens_q, T), pad(enc, lens_k, Lk), pad(dy, lens_q, T)
    causal = torch.full((T, T), NEG, device="cuda").triu(1)[None, None]
    enc_mask = torch.zeros((len(lens_k), 1, 1, Lk), device="cuda")
    for b, n in enumerate(lens_k):
        enc_mask[b, ..., n:] = NEG

    def hf_fwd():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return blk(xp, attention_mask=causal, encoder_hidden_states=ep, encoder_attention_mask=enc_mask)[0]

    def hf_fwd_bwd():
        xh, eh = xp.detach().requires_grad_(True), ep.detach().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = blk(xh, attention_mask=causal, encoder_hidden_states=eh, encoder_attention_mask=enc_mask)[0]
        out.backward(dyp)
        return eh.grad

    fl = flops(lens_q, lens_k)
    res = {"B": len(lens_q), "max_len_q": T, "max_len_k": Lk, **fl}
    res["fwd_ms"] = timed(ours_fwd)
    res["fwd_bwd_ms"] = timed(ours_fwd_bwd)
    res["eager_hf_fwd_ms"] = timed(hf_fwd)
    res["eager_hf_fwd_bwd_ms"] = timed(hf_fwd_bwd)
    for key in ("fwd", "fwd_bwd"):
        res[key + "_tflops"] = fl[key] / res[key + "_ms"] / 1e9
        res[key + "_share_of_datasheet_bf16"] = fl[key] / PEAK_FLOPS * 1e3 / res[key + "_ms"]
        res["speedup_" + key + "_vs_eager_hf"] = res["eager_hf_" + key + "_ms"] / res[key + "_ms"]
    L.profile_enable(True)
    for _ in range(REPS):
        ours_fwd_bwd()
    torch.cuda.synchronize()
    prof = L.profile_report()
    L.profile_enable(False)
    res["kernels"] = {t: {"launches_per_call": r["launches"] / REPS, "ms_per_call": r["ms"] / REPS, "work_per_call": r["work"] / REPS,
                          "tflops": (r["work"] / r["ms"] / 1e9) if t.startswith(("gemm", "attn_fwd", "attn_bwd_dkdv", "attn_bwd_dq")) and r["ms"] > 0 else None}
                      for t, r in prof.items()}
    res["profiled_sum_ms_per_call"] = sum(r["ms"] for r in prof.values()) / REPS
    o = ours_fwd().float()
    h = torch.cat([hf_fwd()[b, :n] for b, n in enumerate(lens_q)]).float()
    res["rel_diff_out_vs_eager_hf"] = float((o - h).norm() / h.norm())
    print(name, json.dumps(res), file=sys.stderr)
    return res


def run_stack(lens_q, lens_k, table):
    g = torch.Generator(device="cuda").manual_seed(24)
    blocks = []
    for _ in range(N_BLOCKS):
        sd = raw_block(g, o_scale=(3 * N_BLOCKS) ** -0.5)
        blocks.append(td.T5DecoderBlockWeights.from_state_dict(sd, H, EPS))
    final_ln = (1.0 + 0.1 * torch.randn((D,), generator=g, device="cuda")).to(torch.bfloat16).float()
    w = td.T5DecoderWeights(blocks, final_ln, table, EPS)
    cuq, cuk = cu(lens_q), cu(lens_k)
    T, Lk = max(lens_q), max(lens_k)
    x = torch.randn((sum(lens_q), D), generator=g, device="cuda").to(torch.bfloat16)
    enc = torch.randn((sum(lens_k), D), generator=g, device="cuda").to(torch.bfloat16).float()
    dy = torch.randn((sum(lens_q), D), generator=g, device="cuda").to(torch.bfloat16)
    state = {}

    def fwd_bwd():
        ek = enc.detach().requires_grad_(True)
        out = td.t5_decoder_stack(x, ek, cuq, cuk, T, Lk, w)
        out.backward(dy)
        state["out"], state["grad"] = out, ek.grad

    fl = flops(lens_q, lens_k)
    res = {"blocks": N_BLOCKS, "fwd_bwd_ms": timed(fwd_bwd, reps=3)}
    res["fwd_bwd_flops"] = N_BLOCKS * fl["fwd_bwd"]
    res["fwd_bwd_tflops"] = res["fwd_bwd_flops"] / res["fwd_bwd_ms"] / 1e9
    res["fwd_bwd_share_of_datasheet_bf16"] = res["fwd_bwd_flops"] / PEAK_FLOPS * 1e3 / res["fwd_bwd_ms"]
    res["out_rms"] = float(state["out"].float().pow(2).mean().sqrt())
    res["enc_grad_finite"] = bool(torch.isfinite(state["grad"]).all())
    res["peak_mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
    print("stack", json.dumps(res), file=sys.stderr)
    return res


def main():
    assert torch.cuda.is_available(), "bench_t5_decoder_block.py measures on the GPU; there is no CPU path"
    g = torch.Generator(device="cuda").manual_seed(0)
    sd = raw_block(g)
    table = (torch.randn((32, H), generator=torch.Generator().manual_seed(1)) * 0.5).to(torch.bfloat16).cuda()
    w = td.T5DecoderBlockWeights.from_state_dict(sd, H, EPS)
    bias = td.t5_position_bias_by_distance(table)
    blk = hf_block(sd, table)
    out = {"card": card(), "d_model": D, "heads": H, "d_ff": D_FF, "reps": REPS,
           "note": "times from CUDA events over REPS back-to-back calls after 2 warm-up calls; forward = inference (no_grad), forward + "
                   "backward = gradients into the bf16 decoder rows and the fp32 aligner rows; eager HF runs on the zero-padded batch with "
                   "masks and is not charged for padding; per-kernel times come from a separate profiled pass (td_profile_enable: events "
                   "between launches, so they include each kernel's prologue); FLOPs are computed from shapes, not counted"}
    for name, (lq, lk) in shapes().items():
        out[name] = run_block(name, lq, lk, w, bias, blk)
    del blk
    torch.cuda.empty_cache()
    out["stack_cfg2"] = run_stack(*shapes()["cfg2"], table)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
