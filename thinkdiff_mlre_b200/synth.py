"""Synthetic batches of the BASELINE.json configs (SURVEY.md section 8d). Pure torch, no CUDA library: this file is also loaded
by path (``importlib``) from ``bench.py --impl reference``, so that the CPU arm never maps ``libthinkdiff_b200.so``.

cfg 2 / 3 / 5 (ThinkDiff-LVLM): a GLOBAL batch of ``world * seqs_per_gpu`` sequences; kept length ``len_i ~ U{1..max_len}`` (the
injected split point of the reference collater, thinkdiff/datasets/datasets/llava_instruct_dataset_mllama_embed_2.py:114), source
length ``L_i = len_i + 1 + (i mod 32)`` (keeps the collater's ``1 <= split <= L_i - 1`` precondition), bf16 N(0,1) features
``[L_i, din]`` and, for the MSE loss, bf16 N(0,1) targets ``[L_i, d]``. Every sequence has its own generator seed, so a rank can
materialise exactly the sequences it was assigned. Which rank gets which sequences is decided by ``sharding.py``.
"""
from __future__ import annotations

import torch


def global_lengths(num_seqs: int, max_len: int, seed: int) -> torch.Tensor:
    """Kept lengths (int32 [num_seqs]) of the global batch with this seed."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(1, max_len + 1, (num_seqs,), generator=g, dtype=torch.int32)


def lvlm_sequences(indices, lens: torch.Tensor, din: int, d: int, seed: int, with_target: bool = True, truncated: bool = False):
    """Materialise the sequences ``indices`` of the global batch ``(seed, lens)`` back to back.

    Returns ``(flat, src_row_start, lens_local, flat_target | None)`` as host tensors. ``truncated``: the source holds only the
    kept rows of every sample (what ``FlatCollater(truncate_on_host=True)`` ships: the reference collater's ``[:split_point]``
    done in the DataLoader worker), so ``src_row_start = cumsum(lens)``."""
    indices = [int(i) for i in indices]
    keep = lens[indices].to(torch.int32)
    full = keep.to(torch.int64) + (0 if truncated else 1 + (torch.tensor(indices, dtype=torch.int64) % 32))
    start = torch.zeros(len(indices), dtype=torch.int64)
    if len(indices) > 1:
        start[1:] = torch.cumsum(full[:-1], 0)
    rows = int(full.sum())
    flat = torch.empty((rows, din), dtype=torch.bfloat16)
    target = torch.empty((rows, d), dtype=torch.bfloat16) if with_target else None
    for k, i in enumerate(indices):
        g = torch.Generator().manual_seed(seed * 1000003 + i)
        n_full = int(keep[k]) + 1 + i % 32          # the sequence's own stream always covers its full source length
        x = torch.randn((n_full, din), generator=g, dtype=torch.float32)
        s0, n = int(start[k]), int(full[k])
        flat[s0 : s0 + n] = x[:n].to(torch.bfloat16)
        if with_target:
            t = torch.randn((n_full, d), generator=g, dtype=torch.float32)
            target[s0 : s0 + n] = t[:n].to(torch.bfloat16)
    return flat, start, keep, target


def lvlm_batch_tensors(num_seqs: int, max_len: int, din: int, d: int, seed: int, with_target: bool = True, truncated: bool = False):
    """One whole batch of ``num_seqs`` sequences (a single rank's view when the global batch is not sharded)."""
    lens = global_lengths(num_seqs, max_len, seed)
    return lvlm_sequences(range(num_seqs), lens, din, d, seed, with_target, truncated)


EOS_ID = 1  # T5's </s>


def t5_labels(num_seqs: int, vocab_size: int, seed: int, min_len: int = 8, max_len: int = 128) -> torch.Tensor:
    """Seeded caption labels in the tokenizer's layout: int64 ``[num_seqs, T]``, sample i holds ``len_i ~ U{min_len..max_len}`` ids
    (``max_len`` 128 is the reference's ``max_txt_len``), the last one EOS (1), the others ``U{2..vocab_size - 1}``, then -100 up to
    ``T = max len_i`` (what the reference's ``targets.masked_fill(pad, -100)`` leaves)."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(min_len, max_len + 1, (num_seqs,), generator=g)
    T = int(lens.max())
    labels = torch.randint(2, vocab_size, (num_seqs, T), generator=g, dtype=torch.int64)
    pos = torch.arange(T)[None, :]
    labels[pos == lens[:, None] - 1] = EOS_ID
    labels[pos >= lens[:, None]] = -100
    return labels
