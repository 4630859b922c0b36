#!/usr/bin/env python
"""Timing of the aligner training step against the reference's objective (AlignerT5TrainStep: pack -> aligner forward -> 24 frozen
Flan-T5-XXL decoder blocks -> lm_head + CrossEntropyLoss -> backward into the aligner -> FusedAdamW) on one B200, next to eager
PyTorch on the same GPU and batches: an nn.Sequential aligner and transformers' T5ForConditionalGeneration (bf16, frozen, dropout
off, a one-layer encoder that is never run) under bf16 autocast on the zero-padded batch with encoder_outputs, attention_mask and
labels, and torch's fused AdamW.

Workload cfg2: 64 samples, aligner rows U{1..256} at 3584 -> 4096 (synth.py), caption labels from synth.t5_labels (U{8..128} tokens,
EOS last), V = 32128, two distinct batches cycled. The decoder's weights are scripts/bench_t5_decoder_block.py's seeded, residual-
scaled blocks; embedding and head share one seeded matrix (transformers 5.x ties them). FLOPs are computed from shapes:
bench_t5_decoder_block.flops x 24, 6 V d per decoder row for the head, 4 Din D + 6 D^2 per aligner row (no dx GEMM). One JSON line.

    python scripts/bench_t5_objective_step.py > profiles/rNN_t5_objective_step.json
"""
import argparse
import json
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import torch

import bench_t5_decoder_block as blk
import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib as L
from thinkdiff_mlre_b200 import ops
from thinkdiff_mlre_b200.optim import FusedAdamW
from thinkdiff_mlre_b200.synth import t5_labels
from thinkdiff_mlre_b200.train_step import make_reference_optimizer

DIN, D, H, D_FF, N_BLOCKS, V, EPS = 3584, 4096, 64, 10240, 24, 32128, 1e-6
B, MAX_K = 64, 256


def hf_model():
    """The frozen bf16 T5ForConditionalGeneration with bench_t5_decoder_block's seeded blocks (o / wo scaled by 1/sqrt(72))."""
    import transformers

    cfg = transformers.T5Config(vocab_size=V, d_model=D, d_kv=64, d_ff=D_FF, num_layers=1, num_decoder_layers=N_BLOCKS, num_heads=H,
                                relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                                feed_forward_proj="gated-gelu", use_cache=False, layer_norm_epsilon=EPS, tie_word_embeddings=False,
                                decoder_start_token_id=0, pad_token_id=0)
    with torch.device("cuda"):
        model = transformers.T5ForConditionalGeneration(cfg).to(torch.bfloat16).eval()
    g = torch.Generator(device="cuda").manual_seed(24)
    table = (torch.randn((32, H), generator=torch.Generator().manual_seed(1)) * 0.5).to(torch.bfloat16).cuda()
    with torch.no_grad():
        for i, b in enumerate(model.decoder.block):
            sd = blk.raw_block(g, o_scale=(3 * N_BLOCKS) ** -0.5)
            if i == 0:
                sd["layer.0.SelfAttention.relative_attention_bias.weight"] = table
            b.load_state_dict(sd)
        model.decoder.final_layer_norm.weight.copy_(1.0 + 0.1 * torch.randn((D,), generator=g, device="cuda"))
        model.shared.weight.copy_(torch.randn((V, D), generator=g, device="cuda") * 2.0 * D ** -0.5)
        model.lm_head.weight.copy_(model.shared.weight)
    return model.requires_grad_(False)


def batches(n=2):
    out = []
    for seed in range(n):
        fb = td.synthetic_lvlm_batch(B, MAX_K, DIN, D, seed=1 + seed, pin=False, with_target=False)
        labels = t5_labels(B, V, seed=200 + seed).cuda()
        flat_q, lens_q, max_q = td.pack_labels(labels, V)
        dev = (fb.flat.cuda(), fb.src_row_start.cuda(), fb.lens.cuda(), fb.total_rows, fb.l_max, flat_q, lens_q.cuda(), max_q)
        cu = ops.cu_seqlens(dev[2])
        xp, mask = ops.pack_padded(dev[0], dev[1], cu, fb.l_max)
        out.append({"step": dev, "padded": (xp, mask, labels), "lens_k": fb.lens.tolist(), "lens_q": lens_q.tolist()})
    return out


def flops(lens_q, lens_k):
    f = N_BLOCKS * blk.flops(lens_q, lens_k)["fwd_bwd"]
    return f + 6.0 * V * D * sum(lens_q) + (4.0 * DIN * D + 6.0 * D * D) * sum(lens_k)


def timed_steps(fn, bs, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(bs[i % len(bs)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--eager-steps", type=int, default=4)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_t5_objective_step.py measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    model = hf_model()
    weights = td.T5ForDecoderWeights.from_module(model)
    torch.manual_seed(0)
    aligner = td.ThinkDiffAligner(DIN, D).cuda()
    eager = torch.nn.Sequential(torch.nn.Linear(DIN, D), torch.nn.GELU(), torch.nn.Linear(D, D), td.aligner._t5_layer_norm_cls()(D, EPS)).cuda()
    eager.load_state_dict(aligner.state_dict())
    bs = batches()
    res = {"card": blk.card(), "workload": {"samples": B, "din": DIN, "d_model": D, "heads": H, "d_ff": D_FF, "blocks": N_BLOCKS, "vocab": V,
                                            "aligner_rows": [sum(b["lens_k"]) for b in bs], "decoder_rows": [sum(b["lens_q"]) for b in bs]}}

    # ---- eager PyTorch: first step from the shared initial parameters, then the timed steps
    opt_e = make_reference_optimizer(eager)

    def eager_step(b):
        xp, mask, labels = b["padded"]
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = model(encoder_outputs=(eager(xp),), attention_mask=mask, labels=labels).loss
        loss.backward()
        opt_e.step()
        opt_e.zero_grad(set_to_none=True)
        return loss

    eager_first = float(eager_step(bs[0]).detach())
    eager_step(bs[1])
    res["eager_step_ms"] = timed_steps(eager_step, bs, args.eager_steps)
    res["eager_peak_mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
    del model, eager, opt_e
    torch.cuda.empty_cache()

    # ---- ours
    step = td.AlignerT5TrainStep(aligner, weights, FusedAdamW(aligner))
    ours_first = float(step.step_device(*bs[0]["step"]))
    res["loss_first_batch"] = ours_first
    res["eager_loss_first_batch"] = eager_first
    res["rel_loss_diff_vs_eager"] = abs(ours_first - eager_first) / abs(eager_first)
    for i in range(args.warmup):
        step.step_device(*bs[(i + 1) % len(bs)]["step"])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    res["step_ms"] = timed_steps(lambda b: step.step_device(*b["step"]), bs, args.steps)
    res["peak_mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
    enq = []
    for i in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step.step_device(*bs[i % len(bs)]["step"])
        enq.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    res["host_enqueue_ms_per_step"] = statistics.median(enq)
    n0 = L.launch_count
    step.step_device(*bs[0]["step"])
    res["launches_per_step"] = L.launch_count - n0

    rows_k = statistics.mean(sum(b["lens_k"]) for b in bs)
    rows_q = statistics.mean(sum(b["lens_q"]) for b in bs)
    fl = statistics.mean(flops(b["lens_q"], b["lens_k"]) for b in bs)
    res["aligner_tokens_per_s"] = rows_k / res["step_ms"] * 1e3
    res["decoder_tokens_per_s"] = rows_q / res["step_ms"] * 1e3
    res["flops_per_step"] = fl
    res["tflops"] = fl / res["step_ms"] / 1e9
    res["share_of_datasheet_bf16"] = fl / blk.PEAK_FLOPS * 1e3 / res["step_ms"]
    res["eager_tflops"] = fl / res["eager_step_ms"] / 1e9
    res["speedup_vs_eager"] = res["eager_step_ms"] / res["step_ms"]

    # ---- per-tag device times, in a pass of its own
    L.profile_enable(True)
    for i in range(len(bs)):
        step.step_device(*bs[i]["step"])
    torch.cuda.synchronize()
    prof = L.profile_report()
    L.profile_enable(False)
    n = len(bs)
    res["kernels"] = {t: {"launches_per_step": r["launches"] / n, "ms_per_step": r["ms"] / n,
                          "tflops": (r["work"] / r["ms"] / 1e9) if t.startswith(("gemm", "attn_fwd", "attn_bwd_dkdv", "attn_bwd_dq")) and r["ms"] > 0 else None}
                      for t, r in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
    res["profiled_sum_ms_per_step"] = sum(r["ms"] for r in prof.values()) / n
    res["note"] = ("step times from CUDA events over --steps back-to-back steps cycling the batches after --warmup steps; eager runs the "
                   "same batches zero-padded and is not charged for padding; peak_mem_gb is the peak of our timed steps with only our weights "
                   "resident; per-kernel times come from a separate profiled pass (events between launches, so they include each kernel's "
                   "prologue); FLOPs are computed from shapes, not counted; first-batch losses are from the same initial parameters")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
