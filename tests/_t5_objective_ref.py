"""Float64 reference of the reference's objective on PACKED rows -- test infrastructure only, the product path never imports it: the
decoder's inputs from the labels (``_shift_right`` + ``embed_tokens`` per sample), the decoder stack of ``_t5_decoder_block_ref``, the
head and ``CrossEntropyLoss(ignore_index=-100)``. tests/test_t5_objective_cpu.py pins it live to transformers'
``T5ForConditionalGeneration(encoder_outputs=..., attention_mask=..., labels=...).loss`` and its gradient with respect to the encoder
states; tests/test_gpu_t5_objective.py compares the kernels against it.

Weights come as a dict (``weights_from_model``): ``blocks`` (per-block dicts in ``T5Block`` state-dict naming), ``final_ln``, ``embed``,
``lm_head``, ``table`` (block 0's relative attention bias), ``start`` / ``pad`` (token ids), ``n_heads`` and ``eps``."""
from __future__ import annotations

import torch

import _t5_decoder_block_ref as ref
from thinkdiff_mlre_b200.t5 import t5_position_bias_by_distance


def shift_right_packed(labels, cu_q, start: int, pad: int) -> torch.Tensor:
    """Decoder input ids of packed labels: the first row of each sample is ``start``, row r > cu_q[b] is ``labels[r - 1]``, -100 -> pad."""
    ids = labels.clone()
    ids[1:] = labels[:-1]
    for b in range(len(cu_q) - 1):
        if cu_q[b + 1] > cu_q[b]:
            ids[cu_q[b]] = start
    return ids.masked_fill(ids == -100, pad)


def weights_from_model(model, dtype=torch.float64) -> dict:
    """The objective's weights of a transformers ``T5ForConditionalGeneration``, in ``dtype``."""
    dec, cfg = model.decoder, model.config
    return {"blocks": [ref.to(b.state_dict(), dtype) for b in dec.block], "final_ln": dec.final_layer_norm.weight.detach().to(dtype),
            "embed": model.get_input_embeddings().weight.detach().to(dtype), "lm_head": model.lm_head.weight.detach().to(dtype),
            "table": dec.block[0].layer[0].SelfAttention.relative_attention_bias.weight.detach(), "start": cfg.decoder_start_token_id,
            "pad": cfg.pad_token_id, "n_heads": cfg.num_heads, "eps": cfg.layer_norm_epsilon}


def loss(enc, labels, cu_q, cu_k, w: dict) -> torch.Tensor:
    """Mean cross-entropy over the labels that are not -100; ``enc [Mk, d]`` packed with ``cu_k``, ``labels`` int64 [Mq] with ``cu_q``."""
    x = w["embed"][shift_right_packed(labels.cpu(), cu_q, w["start"], w["pad"]).to(w["embed"].device)]
    bias = t5_position_bias_by_distance(w["table"]).to(enc)
    h = ref.stack(x, enc, w["blocks"], w["final_ln"], cu_q, cu_k, w["n_heads"], bias, w["eps"])
    return torch.nn.functional.cross_entropy(h @ w["lm_head"].t(), labels.to(h.device), ignore_index=-100)


def loss_and_grad(enc, labels, cu_q, cu_k, w: dict, dtype=torch.float64):
    """``(loss, d loss / d enc)`` in ``dtype`` from the given (e.g. bf16 / fp32) aligner rows."""
    er = enc.detach().to(dtype).requires_grad_(True)
    lo = loss(er, labels, cu_q, cu_k, w)
    lo.backward()
    return lo.detach(), er.grad
