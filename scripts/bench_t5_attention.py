#!/usr/bin/env python
"""Timing of the T5 decoder's attention core on packed rows (SURVEY section 8 f-1; csrc/attn_sm100.cuh) on one B200, forward and
forward + backward, next to two eager baselines on the same GPU and inputs: the HF expression on the padded batch (matmul, + bias /
mask, fp32 softmax, matmul under bf16 autocast, with autograd) and F.scaled_dot_product_attention(scale=1.0) with a float mask.

Shapes (Flan-T5-XXL: 64 heads of d_kv 64): cfg2 cross B = 64, T_b ~ U{8..128}, L_b ~ U{1..256}; cfg5 cross B = 128, L_b ~ U{1..1024};
cfg2 self at the cfg2 decoder lengths. FLOPs count visible (query, key) pairs only: 4 x 64 H per pair forward, 10 x 64 H backward
(the five products of the standard attention backward). HBM bytes: Q, K, V, O (+ LSE) once forward; Q, K, V, O, dO, LSE, Delta read
and dQ, dK, dV written backward. One JSON line on stdout.

    python scripts/bench_t5_attention.py > profiles/rNN_t5_attention.json
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib as L

H, DK = 64, 64
INNER = H * DK
PEAK_FLOPS, PEAK_BYTES = 2250e12, 7.7e12  # B200 data sheet, dense bf16 / HBM3e (1000 W card)
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


def pad(x, cu, n):
    out = x.new_zeros((len(cu) - 1, n, x.shape[1]))
    for b in range(len(cu) - 1):
        out[b, : cu[b + 1] - cu[b]] = x[cu[b] : cu[b + 1]]
    return out.view(len(cu) - 1, n, H, DK).transpose(1, 2)  # [B, H, n, dk]


def unpad(xp, cu):
    x = xp.transpose(1, 2).reshape(xp.shape[0], xp.shape[2], INNER)
    return torch.cat([x[b, : cu[b + 1] - cu[b]] for b in range(len(cu) - 1)])


def run_shape(name, B, t_range, l_range, self_attention, gen):
    lens_q = torch.randint(t_range[0], t_range[1] + 1, (B,), generator=gen).tolist()
    lens_k = lens_q if self_attention else torch.randint(l_range[0], l_range[1] + 1, (B,), generator=gen).tolist()
    cu_q = [0] + torch.tensor(lens_q).cumsum(0).tolist()
    cu_k = [0] + torch.tensor(lens_k).cumsum(0).tolist()
    cuq = torch.tensor(cu_q, dtype=torch.int32, device="cuda")
    cuk = torch.tensor(cu_k, dtype=torch.int32, device="cuda")
    Mq, Mk, T, Lm = cu_q[-1], cu_k[-1], max(lens_q), max(lens_k)
    g = torch.Generator(device="cuda").manual_seed(B)
    q = (torch.randn((Mq, INNER), generator=g, device="cuda") * 0.25).to(torch.bfloat16)
    k = (torch.randn((Mk, INNER), generator=g, device="cuda") * 0.25).to(torch.bfloat16)
    v = torch.randn((Mk, INNER), generator=g, device="cuda").to(torch.bfloat16)
    do = torch.randn((Mq, INNER), generator=g, device="cuda").to(torch.bfloat16)
    table = (torch.randn((32, H), generator=torch.Generator().manual_seed(1)) * 0.5).to(torch.bfloat16)
    bias = td.t5_position_bias_by_distance(table).cuda() if self_attention else None
    ck = None if self_attention else cuk

    def ours_fwd():
        return td.ops.t5_attention_fwd(q, k, v, cuq, ck, T, Lm, H, bias, need_lse=False)[0]

    def ours_fwd_bwd():
        o, lse = td.ops.t5_attention_fwd(q, k, v, cuq, ck, T, Lm, H, bias)
        return td.ops.t5_attention_bwd(do, q, k, v, o, lse, cuq, ck, T, Lm, H, bias)

    # eager baselines on the padded batch: float mask [B or 1, H or 1, T, L]
    qp, kp, vp, dop = pad(q, cu_q, T), pad(k, cu_k, Lm), pad(v, cu_k, Lm), pad(do, cu_q, T)
    neg = torch.finfo(torch.float32).min
    if self_attention:
        pos = torch.arange(T, device="cuda")
        n = pos[:, None] - pos[None, :]
        mask = bias[:, n.clamp(0, bias.shape[1] - 1)].masked_fill(n < 0, neg)[None]  # [1, H, T, T]
    else:
        mask = torch.zeros((B, 1, 1, Lm), device="cuda")
        for b, nk in enumerate(lens_k):
            mask[b, ..., nk:] = neg

    def hf_expr(qx, kx, vx):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            s = torch.matmul(qx, kx.transpose(3, 2))
            s += mask  # HF: in place on the bf16 scores
            p = F.softmax(s.float(), dim=-1).type_as(s)
            return torch.matmul(p, vx)

    def sdpa(qx, kx, vx):
        return F.scaled_dot_product_attention(qx, kx, vx, attn_mask=mask.to(torch.bfloat16), scale=1.0)

    def with_grad(fn):
        def run():
            qx, kx, vx = (t.detach().requires_grad_(True) for t in (qp, kp, vp))
            fn(qx, kx, vx).backward(dop)
        return run

    res = {"B": B, "mode": "self" if self_attention else "cross", "rows_q": Mq, "rows_k": Mk, "max_len_q": T, "max_len_k": Lm}
    pairs = sum(t * (t + 1) // 2 for t in lens_q) if self_attention else sum(t * n for t, n in zip(lens_q, lens_k))
    res["visible_pairs"] = pairs
    flops_f, flops_b = 4.0 * DK * H * pairs, 10.0 * DK * H * pairs
    bytes_f = 2.0 * INNER * (2 * Mq + 2 * Mk) + 4.0 * H * Mq
    bytes_b = 2.0 * INNER * (3 * Mq + 2 * Mk) + 8.0 * H * Mq + 2.0 * INNER * (Mq + 2 * Mk)
    res["fwd_ms"] = timed(ours_fwd)
    res["fwd_bwd_ms"] = timed(ours_fwd_bwd)
    for key, fl, by in (("fwd", flops_f, bytes_f), ("fwd_bwd", flops_f + flops_b, bytes_f + bytes_b)):
        ms = res[key + "_ms"]
        t_fl, t_by = fl / PEAK_FLOPS * 1e3, by / PEAK_BYTES * 1e3
        res[key + "_tflops"] = fl / ms / 1e9
        res[key + "_bound"] = "flops" if t_fl >= t_by else "hbm"
        res[key + "_share_of_bound"] = max(t_fl, t_by) / ms
        res[key + "_bound_ms"] = {"flops": t_fl, "hbm": t_by}
    L.profile_enable(True)
    for _ in range(REPS):
        ours_fwd_bwd()
    torch.cuda.synchronize()
    prof = L.profile_report()
    L.profile_enable(False)
    res["kernels"] = {t: {"ms_per_launch": r["ms"] / r["launches"], "work_per_launch": r["work"] / r["launches"]} for t, r in prof.items()}
    res["eager_hf_fwd_ms"] = timed(lambda: hf_expr(qp, kp, vp))
    res["eager_hf_fwd_bwd_ms"] = timed(with_grad(hf_expr))
    res["sdpa_fwd_ms"] = timed(lambda: sdpa(qp, kp, vp))
    res["sdpa_fwd_bwd_ms"] = timed(with_grad(sdpa))
    res["speedup_fwd_vs_eager_hf"] = res["eager_hf_fwd_ms"] / res["fwd_ms"]
    res["speedup_fwd_vs_sdpa"] = res["sdpa_fwd_ms"] / res["fwd_ms"]
    res["speedup_fwd_bwd_vs_eager_hf"] = res["eager_hf_fwd_bwd_ms"] / res["fwd_bwd_ms"]
    res["speedup_fwd_bwd_vs_sdpa"] = res["sdpa_fwd_bwd_ms"] / res["fwd_bwd_ms"]
    o = ours_fwd()
    ref = unpad(hf_expr(qp, kp, vp), cu_q)
    res["rel_diff_vs_eager_hf"] = float((o.float() - ref.float()).norm() / ref.float().norm())
    res["faster_than_both"] = min(res["speedup_fwd_vs_eager_hf"], res["speedup_fwd_vs_sdpa"], res["speedup_fwd_bwd_vs_eager_hf"],
                                  res["speedup_fwd_bwd_vs_sdpa"]) > 1.0
    print(name, json.dumps(res), file=sys.stderr)
    return res


def main():
    assert torch.cuda.is_available(), "bench_t5_attention.py measures on the GPU; there is no CPU path"
    gen = torch.Generator().manual_seed(0)
    out = {"card": card(), "heads": H, "d_kv": DK, "reps": REPS,
           "note": "times from CUDA events over REPS back-to-back calls after 3 warm-up calls (inputs stay in L2 where they fit); "
                   "eager baselines run on the zero-padded batch and are not charged for padding or un-padding"}
    out["cfg2_cross"] = run_shape("cfg2_cross", 64, (8, 128), (1, 256), False, gen)
    out["cfg5_cross"] = run_shape("cfg5_cross", 128, (8, 128), (1, 1024), False, gen)
    out["cfg2_self"] = run_shape("cfg2_self", 64, (8, 128), None, True, gen)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
