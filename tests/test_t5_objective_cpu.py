"""CPU checks of the reference's objective on packed rows: ``pack_labels`` against transformers' ``_shift_right`` + ``embed_tokens``,
the float64 packed-row reference of the whole objective against live ``T5ForConditionalGeneration(...).loss`` and its gradient with
respect to the encoder states, ``T5ForDecoderWeights``' constructors and refusals, and the seeded label generator. No GPU."""
import types

import pytest
import torch

import _t5_objective_ref as oref
from thinkdiff_mlre_b200.synth import t5_labels
from thinkdiff_mlre_b200.t5 import T5ForDecoderWeights, pack_labels

transformers = pytest.importorskip("transformers")
D, H, D_FF, V, EPS, START, PAD = 128, 2, 96, 64, 1e-6, 2, 0

# interior -100s (sample 0), an all -100 sample (sample 2: zero rows), a sample ending at the last column (sample 3)
LABELS = torch.tensor([[5, -100, 7, 9, 1, -100, -100, -100],
                       [3, 1, -100, -100, -100, -100, -100, -100],
                       [-100, -100, -100, -100, -100, -100, -100, -100],
                       [4, 8, 12, 16, 20, 24, 28, 1]])


def _model(n_layers=2, seed=0, **kw):
    cfg = transformers.T5Config(vocab_size=V, d_model=D, d_kv=64, d_ff=D_FF, num_layers=1, num_decoder_layers=n_layers, num_heads=H,
                                relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                                feed_forward_proj="gated-gelu", use_cache=False, layer_norm_epsilon=EPS, decoder_start_token_id=START,
                                pad_token_id=PAD, **({"tie_word_embeddings": False} | kw))
    model = transformers.T5ForConditionalGeneration(cfg)
    torch.manual_seed(seed)
    with torch.no_grad():
        for p in model.parameters():
            p.copy_(1.0 + 0.1 * torch.randn(p.shape) if p.dim() == 1 else torch.randn(p.shape) * 0.5 * p.shape[-1] ** -0.5)
    return model.eval().requires_grad_(False)


def _cu(lens):
    return [0] + torch.tensor(lens).cumsum(0).tolist()


def test_pack_labels_reproduces_shift_right_and_embed_tokens_at_every_kept_position():
    model = _model(n_layers=1)
    flat, lens, max_len = pack_labels(LABELS, V)
    assert lens.dtype == torch.int32 and lens.tolist() == [5, 2, 0, 8] and max_len == 8
    assert flat.tolist() == [5, -100, 7, 9, 1, 3, 1, 4, 8, 12, 16, 20, 24, 28, 1]
    cu = _cu(lens.tolist())
    ids = oref.shift_right_packed(flat, cu, START, PAD)
    want_ids = model._shift_right(LABELS)
    want_rows = model.decoder.embed_tokens(want_ids)
    rows = model.get_input_embeddings().weight[ids]
    for b, n in enumerate(lens.tolist()):
        assert torch.equal(ids[cu[b] : cu[b] + n], want_ids[b, :n])
        assert torch.equal(rows[cu[b] : cu[b] + n], want_rows[b, :n])
    assert ids[cu[0] + 2] == PAD  # the decoder input after an interior -100 is the pad token


def test_pack_labels_rejects_ids_outside_the_vocabulary():
    for bad in (V, -1, -99, 10**6):
        labels = LABELS.clone()
        labels[1, 0] = bad
        with pytest.raises(ValueError, match="label ids"):
            pack_labels(labels, V)
    with pytest.raises(TypeError):
        pack_labels(LABELS.int(), V)


def test_pack_labels_of_an_all_ignored_batch_has_no_rows():
    flat, lens, max_len = pack_labels(torch.full((3, 4), -100), V)
    assert flat.numel() == 0 and lens.tolist() == [0, 0, 0] and max_len == 0


@pytest.mark.parametrize("lens_k", [[7, 3, 5, 40], [1, 130, 2, 9]])
def test_reference_objective_equals_hf_loss_and_encoder_gradient(lens_k):
    model = _model()
    B, T = LABELS.shape
    L = max(lens_k)
    g = torch.Generator().manual_seed(sum(lens_k))
    enc = torch.randn((sum(lens_k), D), generator=g)
    cu_k = _cu(lens_k)
    enc_p = torch.zeros((B, L, D))
    mask = torch.zeros((B, L), dtype=torch.long)
    for b, n in enumerate(lens_k):
        enc_p[b, :n] = enc[cu_k[b] : cu_k[b + 1]]
        mask[b, :n] = 1
    enc_p = enc_p.double().requires_grad_(True)
    model = model.double()
    want = model(encoder_outputs=(enc_p,), attention_mask=mask, labels=LABELS).loss
    want.backward()

    flat, lens, _ = pack_labels(LABELS, V)
    lo, d_enc = oref.loss_and_grad(enc, flat, _cu(lens.tolist()), cu_k, oref.weights_from_model(model))
    # (the reference's attention core runs in fp32: about 1e-7 relative)
    assert abs(float(lo) - float(want.detach())) <= 1e-6 * abs(float(want.detach()))
    grad_p = enc_p.grad
    want_g = torch.cat([grad_p[b, :n] for b, n in enumerate(lens_k)])
    assert float((d_enc - want_g).abs().max()) <= 1e-5 * float(want_g.abs().max())
    assert all(not grad_p[b, n:].any() for b, n in enumerate(lens_k))  # pad rows of the encoder states: exactly no gradient
    assert not d_enc[cu_k[2] : cu_k[3]].any()  # the sample without decoder rows contributes nothing


def test_weights_from_a_live_model_and_its_state_dict():
    model = _model()
    for w in (T5ForDecoderWeights.from_module(model), T5ForDecoderWeights.from_state_dict(model.state_dict(), model.config)):
        assert len(w.decoder.blocks) == 2 and w.vocab_size == V
        assert (w.decoder_start_token_id, w.pad_token_id) == (START, PAD)
        assert w.embed.dtype == w.lm_head.dtype == torch.bfloat16 and w.embed.shape == (V, D)
        assert torch.equal(w.embed, model.shared.weight.to(torch.bfloat16))
        assert torch.equal(w.lm_head, model.lm_head.weight.to(torch.bfloat16))
        assert torch.equal(w.decoder.final_ln, model.decoder.final_layer_norm.weight)
    model.lm_head.weight.requires_grad_(True)
    with pytest.raises(NotImplementedError, match="must not require grad"):
        T5ForDecoderWeights.from_module(model)


def test_weights_reject_a_config_that_scales_the_decoder_output():
    model = _model(n_layers=1)
    tied = transformers.T5Config(vocab_size=V, d_model=D, d_kv=64, num_heads=H, tie_word_embeddings=True)
    with pytest.raises(NotImplementedError, match="scales the decoder output"):
        T5ForDecoderWeights.from_state_dict(model.state_dict(), tied)
    # the 4.x spelling: no scale_decoder_outputs, tie_word_embeddings=True scales
    for flags in ({"tie_word_embeddings": True}, {"scale_decoder_outputs": True, "tie_word_embeddings": False}):
        cfg = types.SimpleNamespace(**vars(model.config) | flags)
        if "scale_decoder_outputs" not in flags:
            del cfg.scale_decoder_outputs
        with pytest.raises(NotImplementedError, match="scales the decoder output"):
            T5ForDecoderWeights.from_state_dict(model.state_dict(), cfg)
    model.config.scale_decoder_outputs = True
    with pytest.raises(NotImplementedError, match="scales the decoder output"):
        T5ForDecoderWeights.from_module(model)


def test_weights_reject_token_ids_outside_the_vocabulary():
    model = _model(n_layers=1)
    w = T5ForDecoderWeights.from_module(model)
    with pytest.raises(ValueError, match="pad_token_id"):
        T5ForDecoderWeights(w.decoder, model.shared.weight, model.lm_head.weight, 0, V)


def test_label_generator_is_seeded_and_in_the_tokenizer_layout():
    a, b = t5_labels(64, 32128, seed=3), t5_labels(64, 32128, seed=3)
    assert torch.equal(a, b) and not torch.equal(a, t5_labels(64, 32128, seed=4))
    flat, lens, max_len = pack_labels(a, 32128)
    assert a.shape == (64, max_len) and 8 <= int(lens.min()) and max_len <= 128
    for row, n in zip(a, lens.tolist()):
        assert row[n - 1] == 1 and bool((row[: n - 1] >= 2).all()) and bool((row[n:] == -100).all())
