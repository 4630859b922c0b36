#!/usr/bin/env python
"""Benchmark of the ThinkDiff aligner training step (BASELINE.json metric: aligner train tokens/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg5|cfg4]       # this repo's sm_100a path
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   # N > 1
    python bench.py --impl reference ...                                  # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR      # also write the last timed step's outputs (.npy) to compare two builds

One step (cfg2 / cfg5) = pack (features, ragged -> cu_seqlens) -> aligner forward (bf16 autocast regime) -> masked MSE against T5
targets -> aligner backward -> gradient exchange between ranks when N > 1 -> AdamW, on one batch of synthetic Qwen2-VL-7B
features. cfg2: BASELINE config 2 per GPU (64 sequences, valid length U{1..256}, 3584 -> 4096); N GPUs = 64 sequences per rank
(weak scaling; N = 8 is config 3's global batch of 512). cfg5: BASELINE config 5 per GPU (128 sequences, length U{1..1024}).
cfg4: BASELINE config 4 per GPU (inference: 32 samples x two images -> 2 x 32 Q-Former tokens -> aligner -> ragged composition with
T5 text embeddings -> padded prompt). A token = one valid (unpadded) row.

The JSON line: `value` = tokens/s with inputs resident in HBM (CUDA events, max over ranks); `e2e` = the same step fed from pinned
host buffers through the public API, H2D copies and a D2H read of the loss inside the timed region; `roofline` = the dominant
kernel (largest share of device time) from per-launch CUDA events in a separate profiled pass of the same steps; `cpu_baseline` =
the oracle's port of the reference module on this box's host cores; `eager_bar` = the reference module itself (eager PyTorch,
bf16 autocast, cuBLASLt) on this GPU, the same-box bar; `dp_parity` (N > 1) = a numerical check of the multi-GPU path.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

D = 4096
WORKLOADS = {
    # name: (din, sequences per GPU, max valid length, distinct batches cycled)
    "cfg2": (3584, 64, 256, 4),
    "cfg5": (3584, 128, 1024, 1),  # one batch is 1 GB of features + targets: far beyond the 126 MB L2 on its own
    "cfg4": (768, 32, 128, 4),
}
METRIC, UNIT = "aligner_train_tokens_per_sec", "tokens/s"


def flop_per_token(din):
    return 4 * din * D + 6 * D * D  # fwd 2 GEMMs + bwd 3 GEMMs (no dx), SURVEY.md section 8d


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "sm_max_mhz": p.get("sm_max_mhz"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0, "source": "fallback"}


DUMP_SAMPLE = 1 << 22  # entries kept of a larger output array: at most 16 MB per file
DUMP_LIMIT = 64 << 20  # bytes of one whole dump


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write ``arrays`` ({name: tensor}) as ``out_dir/<name>.npy`` in float32, so that two builds of the project can be compared
    output for output from the same command line. An array of more than DUMP_SAMPLE entries is flattened and written as a fixed
    sample of them: sorted flat indices drawn by a generator seeded with the array's size, the same on every run. A set of arrays
    that would take more than DUMP_LIMIT bytes is refused before anything is written."""
    import numpy as np

    total = sum(4 * min(t.numel(), DUMP_SAMPLE) for t in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the limit of {DUMP_LIMIT}")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.RandomState(a.size % (1 << 32)).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_synth():
    """The synthetic generator, loaded by PATH: importing the package would map libthinkdiff_b200.so, which the CPU arm must not."""
    spec = importlib.util.spec_from_file_location("td_synth", os.path.join(ROOT, "thinkdiff_mlre_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ----------------------------------------------------------------------------------------------- clocks
def nvml_handle(pynvml, cuda_index: int):
    """NVML handle of CUDA device `cuda_index` of this process. NVML enumerates every GPU of the box while CUDA enumerates
    CUDA_VISIBLE_DEVICES, so the two indices differ on a shared box: match by UUID (then PCI bus id), index only as a last resort."""
    try:
        import torch

        props = torch.cuda.get_device_properties(cuda_index)
        uuid = getattr(props, "uuid", None)
        if uuid is not None:
            try:
                return pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                pass
        bus = getattr(props, "pci_bus_id", None)
        if bus is not None:
            dom, dev = getattr(props, "pci_domain_id", 0), getattr(props, "pci_device_id", 0)
            return pynvml.nvmlDeviceGetHandleByPciBusId(f"{dom:08x}:{bus:02x}:{dev:02x}.0".encode())
    except Exception:
        pass
    return pynvml.nvmlDeviceGetHandleByIndex(cuda_index)


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while a timed region runs."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = nvml_handle(pynvml, index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # NVML missing: report that instead of guessing
            self.nv, self.err = None, repr(e)
        self.thread = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self._stop.clear()
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *a):
        if self.thread is not None:
            self._stop.set()
            self.thread.join()

    def summary(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": self.err}
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


class numa_local:
    """While active, this process runs on the CPUs NVML reports as local to GPU `index`: pinned host buffers allocated inside
    (first touch) land on the GPU's own NUMA node, so every rank's H2D copies start next to its PCIe root. `cpus` = how many
    CPUs were kept (None: NVML or the affinity call is unavailable, nothing changed)."""

    def __init__(self, index: int):
        self.index, self.cpus, self._saved = index, None, None

    def __enter__(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = nvml_handle(pynvml, self.index)
            words = (os.cpu_count() + 63) // 64
            mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
            cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
            allowed = os.sched_getaffinity(0)
            cpus &= allowed
            if cpus:
                os.sched_setaffinity(0, cpus)
                self._saved, self.cpus = allowed, len(cpus)
        except Exception:
            pass
        return self

    def __exit__(self, *a):
        if self._saved is not None:
            os.sched_setaffinity(0, self._saved)


# ----------------------------------------------------------------------------------------------- CPU reference arm
def cpu_reference_run(steps: int, warmup: int, din: int, seqs: int, max_len: int, max_tokens: int = 2048):
    """The reference's CPU path: the oracle's port of build_vision_projector('mlp2x_gelu_t5_norm') (the reference is
    Python/PyTorch; its own modules cannot travel to the GPU box), fp32, all host threads, on a bounded sample of the
    workload's batch (the first sequences up to `max_tokens` valid tokens): forward + MSE + backward + AdamW."""
    import torch

    from oracle import aligner_ref, pack_ref

    synth = load_synth()
    try:
        cores = len(os.sched_getaffinity(0))  # the CPUs this process may actually run on (a cpuset can be narrower than the machine)
    except (AttributeError, OSError):
        cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    flat, start, lens_t, target = synth.lvlm_batch_tensors(seqs, max_len, din, D, seed=1234)
    lens, keep = lens_t.tolist(), 0
    while keep < len(lens) and sum(lens[: keep + 1]) <= max_tokens:
        keep += 1
    keep = max(keep, 1)
    bits, tbits = flat.view(torch.int16).numpy(), target.view(torch.int16).numpy()
    x, _ = pack_ref.pack_from_flat(bits, start.tolist()[:keep], lens[:keep])      # the collater's job, on the CPU
    t, _ = pack_ref.pack_from_flat(tbits, start.tolist()[:keep], lens[:keep])
    x = torch.from_numpy(x).view(torch.bfloat16).float()
    t = torch.from_numpy(t).view(torch.bfloat16).float()
    m = aligner_ref.RefAligner(din, D)
    m.load_state_dict(aligner_ref.init_params_numpy(din, D, seed=0))
    opt = torch.optim.AdamW(m.parameters(), lr=1e-4, weight_decay=0.05)
    tokens = x.shape[0]

    def step():
        y = m(x)
        loss = torch.nn.functional.mse_loss(y, t)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss.detach()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step()
    dt = time.perf_counter() - t0
    return {"value": tokens * steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {keep} sequences of the batch = {tokens} valid tokens, fp32, fwd+MSE+bwd+AdamW, {steps} steps after {warmup} warm-up",
            "ms_per_step": dt / steps * 1e3, "tokens_per_step": tokens,
            "outputs": {"loss": loss, **{"param." + k: p for k, p in m.named_parameters()}}}


def run_reference_arm(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    din, seqs, max_len, _ = WORKLOADS["cfg2" if args.workload == "cfg4" else args.workload]
    r = cpu_reference_run(args.steps, args.warmup, din, seqs, max_len)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["outputs"])
    line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, args.gpus),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(name, n):
    din, seqs, max_len, nb = WORKLOADS[name]
    what = {"cfg2": "ThinkDiff-LVLM aligner train step (BASELINE config 2 per GPU; N=8 = config 3 global batch 512)",
            "cfg5": "long-context ThinkDiff-LVLM aligner train step (BASELINE config 5 per GPU: 128 sequences, len <= 1024; N=8 = global batch 1024)",
            "cfg4": "ThinkDiff-CLIP two-image + text composition, inference (BASELINE config 4 per GPU: 32 samples; N=8 = batch 256)"}[name]
    cfg = {"workload": what, "name": name, "seqs_per_gpu": seqs, "global_batch": seqs * n, "max_len": max_len, "ragged": f"len ~ U{{1..{max_len}}}",
           "din": din, "d": D, "parallelism": f"dp{n}",
           "sharding": "one global batch of global_batch sequences per step; " + ("length-balanced assignment to ranks (equal sequence counts, even token counts)" if n > 1 else "single rank"),
           "l2_policy": (f"{nb} distinct input batches cycled; " if nb > 1 else "one input batch; ") + "the per-step working set (inputs + activations) exceeds the 126 MB L2"}
    if name != "cfg4":
        cfg.update(loss="masked_mse", optimizer="AdamW wd=0.05")
    return cfg


# ----------------------------------------------------------------------------------------------- eager bar (same box)
def eager_bar(dev, din, seqs, max_len, nb, steps, warmup, rank_seed):
    """The kernel-level bar on the same GPU (SURVEY 8d): the reference's aligner as the reference runs it -- eager
    nn.Sequential(Linear, GELU, Linear, T5LayerNorm) under bf16 autocast on the ZERO-PADDED [B, L_max, Din] batch
    (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:58-63, :585; collater padding ...mllama_embed_2.py:124-127), masked MSE
    on the valid rows, backward(), torch fused AdamW (runners/runner_base.py:122-127): cuBLASLt GEMMs + unfused ATen kernels, no
    kernel of this repo. Also with the packed rows as input (same module, no pad rows). Same batches, same token accounting."""
    import torch
    from torch import nn

    synth = load_synth()
    try:
        from transformers.models.t5.modeling_t5 import T5LayerNorm as Norm
    except Exception:
        class Norm(nn.Module):  # transformers' T5LayerNorm.forward, restated
            def __init__(self, d, eps=1e-6):
                super().__init__()
                self.weight, self.variance_epsilon = nn.Parameter(torch.ones(d)), eps

            def forward(self, h):
                var = h.to(torch.float32).pow(2).mean(-1, keepdim=True)
                h = h * torch.rsqrt(var + self.variance_epsilon)
                if self.weight.dtype in (torch.float16, torch.bfloat16):
                    h = h.to(self.weight.dtype)
                return self.weight * h

    out = {}
    for layout in ("padded", "packed"):
        torch.manual_seed(0)
        model = nn.Sequential(nn.Linear(din, D), nn.GELU(), nn.Linear(D, D), Norm(D)).to(dev)
        decay = [p for n, p in model.named_parameters() if p.ndim >= 2]
        no_decay = [p for n, p in model.named_parameters() if p.ndim < 2]
        opt = torch.optim.AdamW([{"params": decay, "weight_decay": 0.05}, {"params": no_decay, "weight_decay": 0.0}], lr=1e-4, fused=True)
        batches = []
        for j in range(nb):
            flat, start, lens_t, target = synth.lvlm_batch_tensors(seqs, max_len, din, D, seed=rank_seed + 1000 * j)
            lens, l_max = lens_t.tolist(), int(lens_t.max())
            x = torch.zeros((seqs, l_max, din), dtype=torch.bfloat16)
            t = torch.zeros((seqs, l_max, D), dtype=torch.bfloat16)
            mask = torch.zeros((seqs, l_max), dtype=torch.bool)
            for i, (s, n) in enumerate(zip(start.tolist(), lens)):  # the reference collater's pad / stack / mask
                x[i, :n], t[i, :n], mask[i, :n] = flat[s : s + n], target[s : s + n], True
            if layout == "packed":
                batches.append((x[mask].to(dev), t[mask].to(dev), None, int(lens_t.sum())))
            else:
                batches.append((x.to(dev), t.to(dev), mask.to(dev), int(lens_t.sum())))

        def step(x, t, mask, _):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = model(x)
            if mask is None:
                loss = torch.nn.functional.mse_loss(y.float(), t.float())
            else:
                loss = torch.nn.functional.mse_loss(y[mask].float(), t[mask].float())
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return loss

        for i in range(max(warmup, 3)):
            step(*batches[i % nb])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tokens = 0
        e0.record()
        for i in range(steps):
            step(*batches[i % nb])
            tokens += batches[i % nb][3]
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        out[layout] = {"value": tokens / (ms * 1e-3), "ms_per_step": ms / steps}
        del model, opt, batches
        torch.cuda.empty_cache()
    return {"value": out["padded"]["value"], "unit": UNIT, "ms_per_step": out["padded"]["ms_per_step"], "steps": steps,
            "what": "reference nn.Sequential aligner, eager PyTorch under bf16 autocast on the zero-padded batch + masked MSE + backward + torch fused AdamW (cuBLASLt + ATen), same GPU, same batches",
            "packed_rows_variant": {"value": out["packed"]["value"], "ms_per_step": out["packed"]["ms_per_step"],
                                    "what": "same module fed the packed valid rows (no pad rows computed)"}}


# ----------------------------------------------------------------------------------------------- multi-GPU parity
def dp_parity_check(td, dist, dev, world, rank, mode):
    """Numerical check of the multi-GPU path bench.py times, on small dims, outside the timed region:
    (a) the sharded / peer pipelined run == a REPLICATED FusedAdamW run whose gradient is the mean of the per-rank gradients summed
        in rank order (the order the peer path's owners use). Expected: bit-identical parameters after K steps for `peer`; for the
        NCCL `sharded` mode the summation order is NCCL's, and since bf16 training amplifies a 1e-7 difference of an fp32 master
        into 1e-3 of the next gradient, that mode is held to a relative Frobenius distance of 2e-4 instead.
    (b) the exchanged gradient of one step == the mean over ranks of the per-rank gradients of an eager fp32-master / bf16-autocast
        PyTorch aligner on each rank's own shard (DDP's mean of per-rank means, runner_base.py:90-92; <= 2e-2),
    (c) every replica holds bit-identical parameters."""
    import torch
    from torch import nn

    din, d, seqs, max_len, steps = 192, 512, 4, 50, 3
    torch.manual_seed(11)
    ref_sd = {k: v.clone() for k, v in td.ThinkDiffAligner(din, d).to(dev).state_dict().items()}

    def inputs(j):
        b = td.synthetic_lvlm_batch(seqs, max_len, din, d, seed=100 + j, pin=False, world=world, rank=rank)
        cu = td.ops.cu_seqlens(b.lens.to(dev))
        x, idx = td.ops.pack_varlen(b.flat.to(dev), b.src_row_start.to(dev), cu, b.total_rows, want_index=True)
        return b, x, idx, b.extras["flat_target"].to(dev)

    # the path under test
    m = td.ThinkDiffAligner(din, d).to(dev)
    m.load_state_dict(ref_sd)
    m.enable_data_parallel(defer_wait=True, sharded=True, peer=mode == "peer")
    step = td.AlignerTrainStep(m, td.FusedAdamW(m, lr=1e-3), pipelined=True)
    for j in range(steps):
        b, _, _, tgt = inputs(j)
        step.step_device(b.flat.to(dev), b.src_row_start.to(dev), b.lens.to(dev), b.total_rows, b.l_max, tgt)
    step.flush()
    torch.cuda.synchronize()
    tested = [p.detach().clone() for p in m.parameters()]
    if m._peer is not None:
        m._peer.close()  # (collective: nobody still stores into a buffer that is about to be unmapped)

    # (a) replicated AdamW on the rank-ordered mean gradient
    m2 = td.ThinkDiffAligner(din, d).to(dev)
    m2.load_state_dict(ref_sd)
    opt2 = td.FusedAdamW(m2, lr=1e-3)
    inv_world = torch.full((1,), 1.0 / world, dtype=torch.float32, device=dev)
    for j in range(steps):
        _, x, idx, tgt = inputs(j)
        m2.mse_loss_backward_packed(x, tgt, idx, upstream=inv_world)  # this rank's gradient, already divided by the world size
        for name in ("linear1", "linear2"):
            flat = m2._grad_flats[name]
            parts = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(parts, flat)
            acc = parts[0].clone()
            for r in range(1, world):
                acc += parts[r]
            flat.copy_(acc)
        opt2.step()
        opt2.zero_grad()
    torch.cuda.synchronize()
    max_rel, num, den = 0.0, 0.0, 0.0
    for a, t in zip(m2.parameters(), tested):
        max_rel = max(max_rel, float((a.detach() - t).abs().max() / (a.detach().abs().max() + 1e-30)))
        num += float((a.detach() - t).float().pow(2).sum())
        den += float(a.detach().float().pow(2).sum())
    frob = (num / (den + 1e-30)) ** 0.5
    # (c) replicas identical
    replicas_equal = True
    for p in tested:
        ref = p.clone()
        dist.broadcast(ref, src=0)
        replicas_equal = replicas_equal and bool(torch.equal(ref, p))
    flag = torch.tensor([1.0 if replicas_equal else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    replicas_equal = bool(flag.item() == 1.0)
    # (b) one step's exchanged gradient vs the eager PyTorch reference module, mean over ranks
    m3 = td.ThinkDiffAligner(din, d).to(dev)
    m3.load_state_dict(ref_sd)
    m3.enable_data_parallel()
    _, x, idx, tgt = inputs(7)
    m3.mse_loss_backward_packed(x, tgt, idx)
    torch.cuda.synchronize()
    ours = [p.grad.detach().float().clone() for p in m3.parameters()]
    eager = nn.Sequential(nn.Linear(din, d), nn.GELU(), nn.Linear(d, d), type(m3[3])(d, 1e-6)).to(dev)
    eager.load_state_dict(ref_sd)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = eager(x)
    torch.nn.functional.mse_loss(y.float(), tgt[idx].float()).backward()
    grad_rel = 0.0
    for g, p in zip(ours, eager.parameters()):
        r = p.grad.detach().float().clone()
        dist.all_reduce(r)
        r /= world
        grad_rel = max(grad_rel, float((g - r).norm() / (r.norm() + 1e-30)))
    # peer: the owners sum the per-rank slots in rank order, like the reference run here, so the result is bit-identical unless a
    # GEMM's stream-K tail cut different tiles (the scattered GEMMs walk the tiles in a rank-rotated order): allow that last-place
    # difference, amplified by bf16 training as in the NCCL mode
    same = (max_rel == 0.0 or frob <= 2e-4) if mode == "peer" else frob <= 2e-4
    res = {"ok": bool(same and grad_rel <= 2e-2 and replicas_equal), "mode": mode,
           "max_rel_vs_replicated_adamw_on_rank_ordered_mean": max_rel, "frobenius_rel": frob,
           "criterion": "bit-identical, or frobenius_rel <= 2e-4 where a stream-K tail cut different tiles" if mode == "peer" else "frobenius_rel <= 2e-4 (NCCL's summation order differs; bf16 training amplifies 1e-7)",
           "bit_identical": max_rel == 0.0,
           "grad_rel_vs_eager_mean_of_ranks": grad_rel, "replicas_equal": replicas_equal, "steps": steps, "dims": [din, d]}
    del m, m2, m3, eager
    return res


# ----------------------------------------------------------------------------------------------- shard-fed e2e (f-2)
def e2e_from_shards(td, stepper, host_t, seqs, din, dev, steps, sync_all, max_over_ranks, sum_over_ranks, rank):
    """The host-fed step with its batches coming from disk: the synthetic samples are written once as two flat shards (features
    [*, din] and T5-space targets [*, D]; the on-disk format of thinkdiff_mlre_b200/shards.py that replaces the reference's
    pickled tensors in tar shards, thinkdiff/tasks/image_text_process_data.py:94-118), then every step reads its batch with
    EmbedShardReader (one slab copy page cache -> pinned ring buffer, shared by the reader's CPU-bound copy threads), ships it and
    trains on it. The reader is called from this process's main thread between two steps (no background prefetch), so the loader's
    time adds to the step -- it is here to exercise the loader on the GPU path, not to show its best case."""
    import tempfile

    import torch

    tmp = tempfile.mkdtemp(prefix=f"td_shards_r{rank}_")
    paths = (os.path.join(tmp, "feat.tdemb"), os.path.join(tmp, "tgt.tdemb"))
    with td.EmbedShardWriter(paths[0], din) as wf, td.EmbedShardWriter(paths[1], D) as wt:
        for b in host_t:
            for s0, n in zip(b.src_row_start.tolist(), b.lens.tolist()):
                wf.add(b.flat[s0 : s0 + n], [0] * n)
                wt.add(b.extras["flat_target"][s0 : s0 + n], [0] * n)
    rf, rt = td.EmbedShardReader(paths[0]), td.EmbedShardReader(paths[1])
    bi = dict(use_output_embed=1, use_input_embed=0, random_split_output_embed=0, output_embed_max_len=1 << 30, input_embed_max_len=1 << 30)
    nb = len(host_t)

    def load(j):
        fb = rf.batch(j * seqs, (j + 1) * seqs, bi)
        tb = rt.batch(j * seqs, (j + 1) * seqs, bi)
        cbs = [x.extras.get("_h2d_enqueued") for x in (fb, tb)]
        fb.extras["flat_target"] = tb.flat
        fb.extras["_h2d_enqueued"] = lambda evs: [cb(evs) for cb in cbs if cb is not None]
        return fb

    for j in range(2):
        float(stepper.step_prefetched(stepper.prefetch(load(j % nb), dev)))
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    load_s = 0.0
    nxt = stepper.prefetch(load(0), dev)
    for i in range(steps):
        cur = nxt
        if i + 1 < steps:
            tl = time.perf_counter()
            b = load((i + 1) % nb)
            load_s += time.perf_counter() - tl
            nxt = stepper.prefetch(b, dev)
        float(stepper.step_prefetched(cur))
    stepper.flush(sync_masters=False)
    e1.record()
    sync_all()
    stepper.flush()
    ms = max_over_ranks(e0.elapsed_time(e1))
    tokens = sum_over_ranks(float(sum(host_t[i % nb].total_rows for i in range(steps))))
    rf.close(), rt.close()
    for p_ in paths:
        os.remove(p_)
    os.rmdir(tmp)
    return {"value": tokens / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "loader_ms_per_batch": load_s / max(steps - 1, 1) * 1e3,
            "wall_ms_per_step": (time.perf_counter() - t0) / steps * 1e3,
            "copy_threads": rf.copy_threads,
            "note": "batches read from flat on-disk shards by EmbedShardReader, called from the main thread between steps (one slab copy per tensor into a pinned ring recycled on CUDA events, shared by `copy_threads` CPU-bound threads)"}


# ----------------------------------------------------------------------------------------------- B200 arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-eager-bar", action="store_true")
    ap.add_argument("--from-shards", action="store_true",
                    help="also time the host-fed step with its batches read from flat embedding shards on disk (EmbedShardReader, SURVEY 8 f-2)")
    ap.add_argument("--no-dp-parity", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="all-reduce after backward instead of overlapped")
    ap.add_argument("--no-pipeline", action="store_true", help="apply every parameter update inside its own step, on the compute stream")
    ap.add_argument("--dp", default="auto", choices=["auto", "peer", "sharded", "allreduce"],
                    help="N > 1 gradient exchange: peer = reduce-scatter fused into the weight-gradient GEMM epilogues over NVLink peer memory "
                         "(no collective kernels on the step); sharded = NCCL reduce-scatter + row-sharded AdamW + all-gather; allreduce = NCCL "
                         "bucketed all-reduce + replicated AdamW. auto = peer")
    ap.add_argument("--sharding", default="balanced", choices=["balanced", "contiguous"],
                    help="N > 1: how the global batch of N x seqs_per_gpu sequences is split over the ranks -- balanced = equal sequence counts and "
                         "even token counts (SURVEY 8e allows it; synchronous data parallel runs at the pace of the rank with the most tokens), "
                         "contiguous = rank r takes sequences [r * seqs, (r + 1) * seqs)")
    ap.add_argument("--profile-out", default="", help="write the per-kernel table (JSON) here")
    ap.add_argument("--timeline-out", default="", help="write a per-stream device timeline of a few steady-state steps (JSON) here")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused: this repo's one-pass AdamW (+ bf16 copies, per-bucket overlap); torch: torch.optim.AdamW(fused=True)")
    ap.add_argument("--loss-path", default="fused", choices=["fused", "module"],
                    help="fused: fused norm + MSE + norm backward (y/dy stay on chip); module: forward() -> masked MSE -> backward()")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): the loss and every "
                         "parameter after its update (cfg4: the padded prompt embeddings and their mask; --impl reference: the CPU "
                         f"arm's loss and parameters); arrays of more than {DUMP_SAMPLE} entries as a fixed sample of them")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE line (the JSON); anything a library prints there meanwhile (e.g. NCCL's version
    # banner) is diverted to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    # Watchdog: a stream that waits on a peer counter (cuStreamWaitValue32 has no timeout) or a collective whose partner died would
    # otherwise sit there until the launcher's own limit. No run of this script takes anywhere near this long.
    limit = float(os.environ.get("TD_BENCH_WATCHDOG_S", "1800"))
    if limit > 0:
        def _abort():
            try:
                os.write(2, f"bench.py watchdog: no result after {limit:.0f} s (rank {os.environ.get('RANK', '0')}): hung peer wait / collective? aborting\n".encode())
            finally:
                os._exit(4)

        watchdog = threading.Timer(limit, _abort)
        watchdog.daemon = True
        watchdog.start()

    if args.impl == "reference":
        return run_reference_arm(args, emit)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    import torch.distributed as dist

    import thinkdiff_mlre_b200 as td
    from thinkdiff_mlre_b200 import _lib as L
    from thinkdiff_mlre_b200.train_step import make_reference_optimizer

    if world != max(args.gpus, 1) and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch N>1 with torch.distributed.run", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    elif args.dp in ("peer", "sharded"):  # developer aid: the multi-GPU code path degenerated to one rank
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29577")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    warmup = max(args.warmup, 3)
    steps = args.steps
    din, seqs, max_len, num_batches = WORKLOADS[args.workload]
    peaks = measured_peaks()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t)

    if args.workload == "cfg4":
        return run_cfg4(args, emit, td, L, dev, world, rank, local, sync_all, max_over_ranks, sum_over_ranks, peaks)

    torch.manual_seed(0)  # identical init on every rank (DDP broadcasts rank 0's; same seed is equivalent)
    aligner = td.ThinkDiffAligner(din, D).to(dev)
    fused = args.optimizer == "fused" and args.loss_path == "fused"
    pipelined = fused and not args.no_pipeline
    dp_mode, dp_fallback = None, None
    if world > 1 or args.dp in ("peer", "sharded"):
        dp_mode = "peer" if args.dp == "auto" else args.dp
        if not (pipelined and D % world == 0) and dp_mode in ("peer", "sharded"):
            dp_mode = "allreduce"
        aligner.enable_data_parallel(overlap=not args.no_overlap, defer_wait=args.optimizer == "fused", sharded=dp_mode in ("sharded", "peer"),
                                     peer=dp_mode == "peer")
        if dp_mode == "peer":
            # map the exchange buffers now (collective). `--dp auto`: a box without peer access / CUDA IPC falls back to the NCCL
            # row-sharded exchange on every rank (the set-up fails on all ranks or on none) and the line says so.
            from thinkdiff_mlre_b200.peer import PeerSetupError

            try:
                aligner._ensure_peer()
            except PeerSetupError as e:
                if args.dp != "auto":
                    raise
                dp_fallback = str(e)[:300]
                dp_mode = "sharded"
                aligner.enable_data_parallel(overlap=not args.no_overlap, defer_wait=True, sharded=True, peer=False)
    opt = td.FusedAdamW(aligner, lr=1e-4, weight_decay=0.05) if args.optimizer == "fused" else make_reference_optimizer(aligner)
    stepper = td.AlignerTrainStep(aligner, opt, fused_loss=args.loss_path == "fused", pipelined=pipelined)

    with numa_local(local) as numa:
        host = [td.synthetic_lvlm_batch(seqs, max_len, din, D, seed=1234 + 1000 * j, world=world, rank=rank, balanced=args.sharding == "balanced")
                for j in range(num_batches)]
    numa_cpus = numa.cpus
    resident = [(b.flat.to(dev), b.src_row_start.to(dev), b.lens.to(dev), b.total_rows, b.l_max, b.extras["flat_target"].to(dev)) for b in host]
    tokens_per_step = [b.total_rows for b in host]

    # ---- device-resident timing ------------------------------------------------------------------
    for i in range(warmup):
        stepper.step_device(*resident[i % num_batches])
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = L.launch_count
    clocks = ClockSampler(local)
    with clocks:
        e0.record()
        t_host0 = time.perf_counter()
        for i in range(steps):
            loss = stepper.step_device(*resident[i % num_batches])
        host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / steps  # CPU time to enqueue one step (no sync inside)
        # pipelined mode: the last step's parameter updates (AdamW + exchange of the bf16 rows) are part of the timed work; the
        # all-gather of the other ranks' fp32 MASTER rows, which only a checkpoint needs, is done after the timed region
        stepper.flush(sync_masters=False)
        e1.record()
        sync_all()
    stepper.flush()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = L.launch_count - launches0
    tokens = sum_over_ranks(float(sum(tokens_per_step[i % num_batches] for i in range(steps))))
    value = tokens / (ms * 1e-3)
    final_loss = float(loss)
    if args.dump_outputs and rank == 0:  # before the passes below train the aligner further
        dump_outputs(args.dump_outputs, {"loss": loss, **{"param." + k: p for k, p in aligner.named_parameters()}})

    # ---- end to end: pinned host buffers -> H2D -> step -> D2H loss, every step ---------------------
    e2e = None
    if not args.no_e2e:
        # what the collater ships: only the kept rows of every sample (FlatCollater(truncate_on_host=True), the reference
        # collater's [:split_point] done in the DataLoader worker) -- the device pack then re-packs contiguous rows
        with numa_local(local):
            host_t = [td.synthetic_lvlm_batch(seqs, max_len, din, D, seed=1234 + 1000 * j, truncated=True, world=world, rank=rank,
                                              balanced=args.sharding == "balanced") for j in range(num_batches)]
        for i in range(3):
            float(stepper.step_host(host_t[i % num_batches], dev))
        copy_streams = stepper.tune_copy_streams(host_t[0], dev)  # 1 / 2 / 4 copy streams: whichever this host moves a batch fastest with
        sync_all()
        e0.record()
        nxt = stepper.prefetch(host_t[0], dev)  # inside the timed region: every step's H2D is paid for
        for i in range(steps):
            cur = nxt
            if i + 1 < steps:
                nxt = stepper.prefetch(host_t[(i + 1) % num_batches], dev)  # copy of step i+1 overlaps compute of step i
            loss_host = float(stepper.step_prefetched(cur))  # .item(): D2H read of the loss, as base_task.py:262
        stepper.flush(sync_masters=False)
        e1.record()
        sync_all()
        stepper.flush()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        tokens_e2e = sum_over_ranks(float(sum(host_t[i % num_batches].total_rows for i in range(steps))))
        b0 = host_t[0]
        h2d = b0.flat.nbytes + b0.extras["flat_target"].nbytes + b0.src_row_start.nbytes + b0.lens.nbytes
        e2e = {"value": tokens_e2e / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e / steps, "h2d_gbs_per_rank": h2d / (ms_e2e / steps * 1e-3) / 1e9, "numa_bound_cpus": numa_cpus, "copy_streams": copy_streams,
               "note": "every step: H2D of the kept rows of its bf16 features + T5 targets from pinned memory (row chunks over `copy_streams` copy streams, picked by timing 1 / 2 / 4 on this host before the timed region; overlapping the previous step's compute) and loss.item()"}
        if args.from_shards:
            e2e["from_shards"] = e2e_from_shards(td, stepper, host_t, seqs, din, dev, min(steps, 12), sync_all, max_over_ranks, sum_over_ranks, rank)
        del host_t

    if os.environ.get("TD_HOST_PROFILE") and rank == 0:  # developer aid: where does the host time of a step go?
        import cProfile, io, pstats

        pr = cProfile.Profile()
        pr.enable()
        for i in range(100):
            stepper.step_device(*resident[i % num_batches])
        pr.disable()
        stepper.flush()
        buf = io.StringIO()
        pstats.Stats(pr, stream=buf).sort_stats("tottime").print_stats(22)
        print(buf.getvalue()[:5000], file=sys.stderr)
    elif os.environ.get("TD_HOST_PROFILE"):
        for i in range(100):
            stepper.step_device(*resident[i % num_batches])
        stepper.flush()

    # ---- per-stream device timeline of steady-state steps (same pipelined step the timed region ran) ----------
    if args.timeline_out:
        for i in range(2):
            stepper.step_device(*resident[i % num_batches])
        L.profile_enable(True)
        for i in range(4):
            stepper.step_device(*resident[(i + 2) % num_batches])
        stepper.flush(sync_masters=False)
        sync_all()
        recs = L.profile_timeline()
        L.profile_enable(False)
        stepper.flush()
        streams = sorted({r[1] for r in recs})
        tl = {"rank": rank, "n_gpus": world, "dp": dp_mode, "steps": 4, "unit": "ms since the first recorded launch",
              "streams": {s: i for i, s in enumerate(streams)},
              "launches": [{"tag": r[0], "stream": streams.index(r[1]), "t0": r[2], "t1": r[3]} for r in recs],
              "note": "CUDA events around every launch of this library; events of different streams share the device clock. Gaps on the compute stream are waits (for a parameter update / a peer flag / a collective) or launch gaps."}
        path = args.timeline_out.replace("%r", str(rank))
        if rank == 0 or "%r" in args.timeline_out:
            os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
            with open(path, "w") as f:
                json.dump(tl, f)

    # ---- per-kernel device times (separate pass of the same steps; CUDA events around every launch) --
    psteps = min(steps, 20)
    prof_stepper, profile_pass = stepper, "same pipelined step (kernels of different streams overlap: per-launch times are upper bounds)"
    if world == 1 and pipelined and dp_mode is None:
        # one stream, no overlap between the AdamW side stream and the GEMMs: clean per-kernel times for the roofline
        stepper.flush()
        aligner._bwd_order, aligner._record_phase_events = "linear2_first", False
        prof_stepper = td.AlignerTrainStep(aligner, opt, fused_loss=True, pipelined=False)
        profile_pass = "sequential step: same kernels, same inputs, single stream (the timed region overlaps AdamW with the GEMMs)"
        for i in range(2):
            prof_stepper.step_device(*resident[i % num_batches])
    L.profile_enable(True)
    for i in range(psteps):
        prof_stepper.step_device(*resident[i % num_batches])
    prof_stepper.flush()
    torch.cuda.synchronize()
    prof = L.profile_report()
    L.profile_enable(False)
    clk = clocks.summary()
    at_max_clock = bool(clk.get("sm_mhz") and clk.get("sm_max_mhz") and clk["sm_mhz"] >= 0.97 * clk["sm_max_mhz"])
    # a kernel timed while the SM clock holds its maximum is compared with the burst cuBLAS figure; under the power cap
    # (seconds-long runs) the sustained figure is the comparable one. Both fractions are reported.
    tc_peak = peaks["bf16_tflops"] if at_max_clock else peaks["bf16_tflops_sustained"]
    kernels = {}
    for tag, r in prof.items():
        per_launch_ms = r["ms"] / r["launches"]
        rate = r["work"] / (r["ms"] * 1e-3)
        if tag.startswith("gemm_"):
            kernels[tag] = {"launches_per_step": r["launches"] / psteps, "ms_per_launch": per_launch_ms, "bound": "tensor",
                            "achieved": rate / 1e12, "unit": "TFLOP/s", "frac": rate / 1e12 / tc_peak,
                            "frac_burst": rate / 1e12 / peaks["bf16_tflops"], "frac_sustained": rate / 1e12 / peaks["bf16_tflops_sustained"]}
        else:
            kernels[tag] = {"launches_per_step": r["launches"] / psteps, "ms_per_launch": per_launch_ms, "bound": "hbm",
                            "achieved": rate / 1e9, "unit": "GB/s", "frac": rate / 1e9 / peaks["hbm_gbs"]}
    total_ms = sum(r["ms"] for r in prof.values()) / psteps
    for tag, r in prof.items():
        kernels[tag]["share_of_kernel_time"] = (r["ms"] / psteps) / total_ms
    dom = max(kernels, key=lambda k: kernels[k]["share_of_kernel_time"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # dram bytes per launch from the committed ncu capture
    if os.path.isfile(tpath) and args.workload == "cfg2":
        traffic = json.load(open(tpath)).get(dom)
    roofline = {"kernel": dom, "bound": kernels[dom]["bound"], "achieved": kernels[dom]["achieved"],
                "peak": tc_peak if kernels[dom]["bound"] == "tensor" else peaks["hbm_gbs"],
                "unit": kernels[dom]["unit"], "frac": kernels[dom]["frac"], "traffic": traffic,
                "peak_source": f"MEASURED_PEAKS.json ({peaks['source']}): " + ("burst bf16 figure, the sampled SM clock held its maximum" if at_max_clock else "sustained bf16 figure, the SM clock sagged under the power cap"),
                "frac_burst": kernels[dom].get("frac_burst"), "frac_sustained": kernels[dom].get("frac_sustained"),
                "ms_per_launch": kernels[dom]["ms_per_launch"], "share_of_kernel_time": kernels[dom]["share_of_kernel_time"],
                "profile_pass": profile_pass}

    # ---- N > 1: numerical check of the path that was timed, outside the timed region -------------
    dp_parity = None
    if world > 1 and not args.no_dp_parity and dp_mode in ("peer", "sharded"):
        dp_parity = dp_parity_check(td, dist, dev, world, rank, dp_mode)

    cpu = bar = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(5, 2, din, seqs, max_len)
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if rank == 0 and world == 1 and not args.no_eager_bar:
        del resident
        torch.cuda.empty_cache()
        bar = eager_bar(dev, din, seqs, max_len, num_batches, min(steps, 20), 3, 1234)
        bar["speedup_of_this_repo"] = value / bar["value"]

    ok = True
    if rank == 0:
        step_tflops = value / world * flop_per_token(din) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": dict(workload_config(args.workload, world), loss_path=args.loss_path, optimizer_impl=args.optimizer, pipelined_updates=pipelined,
                                                 dp_exchange=dp_mode, dp_exchange_fallback=dp_fallback, sharding_mode=args.sharding if world > 1 else None, fp32_master_sync="after the timed region (bf16 compute copies and AdamW are inside it)" if dp_mode in ("peer", "sharded") else None),
            "clocks": clk, "e2e": e2e,
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "eager_bar": bar, "dp_parity": dp_parity,
            "step_tflops_per_gpu": step_tflops, "step_frac_of_bf16_peak": step_tflops / tc_peak,
            "step_frac_of_bf16_burst": step_tflops / peaks["bf16_tflops"], "step_frac_of_bf16_sustained": step_tflops / peaks["bf16_tflops_sustained"],
            "step_frac_of_nominal_2250": step_tflops / 2250.0, "tokens_per_step": tokens / steps, "final_loss": final_loss,
            "host_enqueue_ms_per_step": host_enqueue_ms, "kernels": kernels,
        }
        if args.profile_out:
            os.makedirs(os.path.dirname(os.path.abspath(args.profile_out)), exist_ok=True)
            with open(args.profile_out, "w") as f:
                json.dump({"kernels": kernels, "kernel_ms_per_step": total_ms, "ms_per_step": ms / steps, "peaks": peaks}, f, indent=1)
        emit(line)
        ok = dp_parity is None or dp_parity["ok"]
    if dist.is_initialized():
        dist.destroy_process_group()
    if not ok:
        print("bench.py: dp_parity FAILED", dp_parity, file=sys.stderr)
        sys.exit(3)


def run_cfg4(args, emit, td, L, dev, world, rank, local, sync_all, max_over_ranks, sum_over_ranks, peaks):
    """BASELINE config 4 per GPU: inference. Two images per sample -> 2 x 32 Q-Former tokens [768] -> aligner (pure-bf16 regime,
    scripts/test/test_blip_vision_t5_decoder_flux_text.py:104) -> ragged [img1 | img2 | text_i] composition with T5 text embeddings
    (:184-208) -> zero-padded prompt_embeds + int64 mask. Tokens = packed rows (64 + T_i per sample)."""
    import torch

    din, seqs, max_len, nb = WORKLOADS["cfg4"]
    steps, warmup = args.steps, max(args.warmup, 3)
    torch.manual_seed(0)
    aligner = td.ThinkDiffAligner(din, D).to(dev).to(torch.bfloat16).eval()
    batches = []
    for j in range(nb):
        g = torch.Generator().manual_seed(4321 + rank + 1000 * j)
        q = torch.randn((seqs, 64, din), generator=g).to(torch.bfloat16)
        tl = torch.randint(1, max_len + 1, (seqs,), generator=g).tolist()
        text = torch.randn((sum(tl), D), generator=g).to(torch.bfloat16)
        batches.append((q.to(dev), text.to(dev), tl, seqs * 64 + sum(tl)))

    def step(q, text, tl, _):
        with torch.no_grad():
            y = aligner(q)                                  # [B, 64, 4096] bf16
            packed = td.compose_image_text(y, text, tl)     # ragged [64 + T_i] rows
            return packed.to_padded()                       # [B, L_max, 4096] + int64 mask

    for i in range(warmup):
        step(*batches[i % nb])
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = L.launch_count
    clocks = ClockSampler(local)
    with clocks:
        e0.record()
        for i in range(steps):
            out = step(*batches[i % nb])
        e1.record()
        sync_all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"prompt_embeds": out[0], "prompt_mask": out[1]})
    ms = max_over_ranks(e0.elapsed_time(e1))
    tokens = sum_over_ranks(float(sum(batches[i % nb][3] for i in range(steps))))
    L.profile_enable(True)
    for i in range(min(steps, 20)):
        step(*batches[i % nb])
    torch.cuda.synchronize()
    prof = L.profile_report()
    L.profile_enable(False)
    kernels = {}
    for tag, r in prof.items():
        rate = r["work"] / (r["ms"] * 1e-3)
        tensor = tag.startswith("gemm_")
        kernels[tag] = {"launches_per_step": r["launches"] / min(steps, 20), "ms_per_launch": r["ms"] / r["launches"], "bound": "tensor" if tensor else "hbm",
                        "achieved": rate / (1e12 if tensor else 1e9), "unit": "TFLOP/s" if tensor else "GB/s",
                        "frac": rate / (1e12 * peaks["bf16_tflops"] if tensor else 1e9 * peaks["hbm_gbs"])}
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_launch"] * kernels[k]["launches_per_step"])
    if rank == 0:
        emit({"metric": "aligner_compose_tokens_per_sec", "value": tokens / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
              "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
              "config": workload_config("cfg4", world), "clocks": clocks.summary(), "e2e": None, "gpu_launches": L.launch_count - launches0,
              "roofline": {"kernel": dom, "bound": kernels[dom]["bound"], "achieved": kernels[dom]["achieved"], "unit": kernels[dom]["unit"],
                           "peak": peaks["bf16_tflops"] if kernels[dom]["bound"] == "tensor" else peaks["hbm_gbs"], "frac": kernels[dom]["frac"], "traffic": None},
              "cpu_baseline": None, "kernels": kernels, "tokens_per_step": tokens / steps})
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
