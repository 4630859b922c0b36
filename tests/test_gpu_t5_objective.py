"""GPU checks of the reference's objective on packed rows (td_t5_decoder_inputs, td_t5_cross_attention_layer_bwd_accumulate,
ops.t5_decoder_loss_fwd_bwd / t5_decoder_loss, AlignerT5TrainStep): the decoder inputs bit-exact against torch's gather; the
accumulating cross-attention backward exactly fp32(g + d_enc); t5_decoder_loss bit-identical in loss and gradient to the autograd
composition embed -> t5_decoder_stack -> lm_head_cross_entropy; the train step bit-identical to forward_packed + t5_decoder_loss +
backward + the same optimizer, linear in its loss scale, and with the launch count DESIGN states; loss and aligner gradients against
float64 at most 1.25x the error of eager HF (nn.Sequential aligner + T5ForConditionalGeneration) under bf16 autocast."""
import pytest
import torch

import _t5_objective_ref as oref
import thinkdiff_mlre_b200 as td
from thinkdiff_mlre_b200 import _lib, ops
from thinkdiff_mlre_b200.optim import FusedAdamW

pytestmark = pytest.mark.gpu
EPS = 1e-6


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _cu(lens):
    return torch.tensor([0] + torch.tensor(lens).cumsum(0).tolist(), dtype=torch.int32, device="cuda")


def _shift_right(flat, lens, start, pad):
    ids = flat.clone()
    ids[1:] = flat[:-1]
    ids[_cu(lens)[:-1][torch.tensor(lens, device="cuda") > 0].long()] = start
    return ids.masked_fill(ids == -100, pad)


def _labels(lens, V, seed, ignore=0.15):
    """Right-padded [B, T] labels with interior -100s; the last kept position of every non-empty sample is a real id."""
    g = torch.Generator().manual_seed(seed)
    T = max(max(lens), 1)
    lab = torch.randint(0, V, (len(lens), T), generator=g)
    lab[torch.rand((len(lens), T), generator=g) < ignore] = -100
    for b, n in enumerate(lens):
        lab[b, n:] = -100
        if n:
            lab[b, n - 1] = int(torch.randint(0, V, (1,), generator=g))
    return lab.cuda()


def _decoder_weights(d, H, d_ff, n_blocks, V, seed):
    """Seeded frozen objective weights (bf16 values; q / k scaled so scores stay O(1), o / wo by 1/sqrt(3 n_blocks) so the residual
    stream stays O(1)), embed and lm_head separate tensors."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    inner = 64 * H

    def lin(n_out, n_in, s=1.0):
        return (torch.randn((n_out, n_in), generator=g, device="cuda") * s * n_in ** -0.5).to(torch.bfloat16)

    def ln():
        return (1.0 + 0.1 * torch.randn((d,), generator=g, device="cuda")).to(torch.bfloat16).float()

    o_s = (3 * n_blocks) ** -0.5
    blocks = []
    for _ in range(n_blocks):
        ffn = td.T5FeedForwardWeights(lin(d_ff, d), lin(d_ff, d), lin(d, d_ff, o_s), ln(), EPS)
        blocks.append(td.T5DecoderBlockWeights(ln(), lin(inner, d, 0.25), lin(inner, d, 0.25), lin(inner, d), lin(d, inner, o_s), ln(),
                                               lin(inner, d, 0.25), lin(inner, d, 0.25), lin(inner, d), lin(d, inner, o_s), ffn, H, EPS))
    table = (0.5 * torch.randn((32, H), generator=g, device="cuda")).to(torch.bfloat16)
    dec = td.T5DecoderWeights(blocks, ln(), table, EPS)
    return td.T5ForDecoderWeights(dec, lin(V, d, d ** 0.5 * 0.5), lin(V, d, 2.0), decoder_start_token_id=0, pad_token_id=0)


# ------------------------------------------------------------------------------------------------ decoder inputs
@pytest.mark.parametrize("d", [512, 4096])
def test_decoder_inputs_are_embed_of_shift_right_bit_exactly(d):
    V = 32128
    g = torch.Generator(device="cuda").manual_seed(d)
    embed = torch.randn((V, d), generator=g, device="cuda").to(torch.bfloat16)
    for lens in ([0, 1, 7, 0], [1], [63, 64, 65, 0, 128, 1], [8] * 300):
        labels = _labels(lens, V, seed=sum(lens) + d)
        flat, lq, _ = td.pack_labels(labels, V)
        assert lq.tolist() == lens
        rows = ops.t5_decoder_inputs(flat, _cu(lens), embed, 3, 0)
        assert rows.shape == (sum(lens), d)
        assert torch.equal(rows, embed[_shift_right(flat, lens, 3, 0)])
    # more samples than the kernel stages in shared memory (2048)
    lens = [0, 1, 2] * 700 + [5]
    flat, _, _ = td.pack_labels(_labels(lens, V, seed=7), V)
    assert torch.equal(ops.t5_decoder_inputs(flat, _cu(lens), embed, 3, 0), embed[_shift_right(flat, lens, 3, 0)])


def test_decoder_inputs_of_ids_outside_the_table_are_zero_rows():
    V, d = 1000, 512
    embed = torch.randn((V, d), device="cuda").to(torch.bfloat16)
    flat = torch.tensor([5, V, -5, 7, 2**40, -100, 9], dtype=torch.int64, device="cuda")
    rows = ops.t5_decoder_inputs(flat, _cu([4, 3]), embed, V + 3, 1)
    ids = [V + 3, 5, V, -5, V + 3, 2**40, 1]
    for r, i in enumerate(ids):
        want = embed[i] if 0 <= i < V else torch.zeros(d, dtype=torch.bfloat16, device="cuda")
        assert torch.equal(rows[r], want), r
    assert ops.t5_decoder_inputs(flat[:0], _cu([0, 0]), embed, 0, 0).shape == (0, d)


# ------------------------------------------------------------------------------------------------ accumulating cross-attention backward
@pytest.mark.parametrize("d,H", [(512, 8), (4096, 64)])
def test_cross_attention_backward_accumulates_exactly(d, H):
    w = _decoder_weights(d, H, 2 * d, 1, 64, seed=d).decoder.blocks[0]
    lens_q, lens_k = [1, 128, 40], [200, 0, 33]
    cuq, cuk = _cu(lens_q), _cu(lens_k)
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn((sum(lens_q), d), generator=g, device="cuda").to(torch.bfloat16)
    enc = torch.randn((sum(lens_k), d), generator=g, device="cuda").to(torch.bfloat16)
    dy = torch.randn((sum(lens_q), d), generator=g, device="cuda").to(torch.bfloat16)
    _, *saved = ops.t5_cross_attention_layer_fwd(x, enc, w.w_q, w.w_kv, w.wo_cross, w.ln_cross, w.eps, cuq, cuk, 128, 200, H)
    args = (*saved, w.w_q, w.w_kv, w.wo_cross, w.ln_cross, cuq, cuk, 128, 200, H)
    dx0, d0 = ops.t5_cross_attention_layer_bwd(dy, x, *args)
    dx1, d1 = ops.t5_cross_attention_layer_bwd(dy, x, *args)
    assert torch.equal(dx0, dx1) and torch.equal(d0, d1)  # the overwrite form, unchanged and deterministic
    # g ~ N(0, 1) fp32 with |g| >= 2^-20: no subnormal input or sum occurs (a bulk fp32 reduction may flush subnormals)
    acc = torch.randn(d0.shape, generator=g, device="cuda")
    acc = torch.where(acc.abs() < 2.0 ** -20, torch.full_like(acc, 2.0 ** -20), acc)
    want = acc + d0
    assert not bool(((want != 0) & (want.abs() < torch.finfo(torch.float32).tiny)).any())
    buf = acc.clone()
    dx2, out = ops.t5_cross_attention_layer_bwd(dy, x, *args, d_enc_accumulate=buf)
    assert out is buf and torch.equal(dx2, dx0)
    assert torch.equal(buf, want)
    zero = torch.zeros_like(d0)
    ops.t5_cross_attention_layer_bwd(dy, x, *args, d_enc_accumulate=zero)
    assert torch.equal(zero, d0)
    with pytest.raises(TypeError, match="d_enc_accumulate"):
        ops.t5_cross_attention_layer_bwd(dy, x, *args, d_enc_accumulate=buf.to(torch.bfloat16))


# ------------------------------------------------------------------------------------------------ t5_decoder_loss vs the composition
@pytest.mark.parametrize("d,H,n_blocks", [(512, 8, 3), (4096, 64, 2)])
def test_decoder_loss_is_bit_identical_to_the_autograd_composition(d, H, n_blocks):
    V = 32128 if d == 4096 else 512
    w = _decoder_weights(d, H, 2 * d if d == 512 else 10240, n_blocks, V, seed=n_blocks)
    lens_q, lens_k = [17, 0, 128, 1, 65], [40, 9, 256, 0, 3]
    labels = _labels(lens_q, V, seed=5)
    flat, lq, Tq = td.pack_labels(labels, V)
    cuq, cuk, Tk = ops.cu_seqlens(lq.cuda()), _cu(lens_k), max(lens_k)
    enc = torch.randn((sum(lens_k), d), generator=torch.Generator(device="cuda").manual_seed(3), device="cuda")

    ea = enc.clone().requires_grad_(True)
    rows = w.embed[_shift_right(flat, lq.tolist(), w.decoder_start_token_id, w.pad_token_id)]
    loss_a = td.lm_head_cross_entropy(td.t5_decoder_stack(rows, ea, cuq, cuk, Tq, Tk, w.decoder), w.lm_head, flat)
    loss_a.backward()

    eb = enc.clone().requires_grad_(True)
    loss_b = td.t5_decoder_loss(eb, cuk, Tk, flat, cuq, Tq, w)
    loss_b.backward()
    assert torch.equal(loss_a, loss_b)
    assert eb.grad.dtype == torch.float32 and torch.equal(ea.grad, eb.grad)
    assert not eb.grad[40:49].any()  # the aligner rows of the sample without decoder rows get exactly no gradient

    with torch.no_grad():  # the forward only: same loss
        assert torch.equal(td.t5_decoder_loss(eb, cuk, Tk, flat, cuq, Tq, w), loss_b)
    # the cross-entropy kernel folds grad_scale into its softmax exponent (log2(scale / sum)): linear up to the rounding it moves
    loss_s, d_s = ops.t5_decoder_loss_fwd_bwd(enc, cuk, Tk, flat, cuq, Tq, w, grad_scale=4.0)
    assert torch.equal(loss_s, loss_b) and _rel(d_s, 4.0 * eb.grad) < 1e-3


# ------------------------------------------------------------------------------------------------ the train step
DIN, D, H, NB, V = 256, 512, 8, 2, 512


def _aligner(seed):
    torch.manual_seed(seed)
    a = td.ThinkDiffAligner(DIN, D).cuda()
    with torch.no_grad():
        a[3].weight.copy_(1.0 + 0.1 * torch.randn(D))
    return a


def _batch(seed, n=6):
    b = td.synthetic_lvlm_batch(n, 200, DIN, D, seed=seed, pin=False, with_target=False)
    lens_q = torch.randint(8, 129, (n,), generator=torch.Generator().manual_seed(seed)).tolist()
    flat_q, lq, Tq = td.pack_labels(_labels(lens_q, V, seed), V)
    return (b.flat.cuda(), b.src_row_start.cuda(), b.lens.cuda(), b.total_rows, b.l_max, flat_q, lq.cuda(), Tq)


def test_train_step_matches_autograd_and_fused_adamw_bit_for_bit():
    w = _decoder_weights(D, H, 1024, NB, V, seed=21)
    batches = [_batch(1), _batch(2)]
    a, b = _aligner(0), _aligner(0)
    step = td.AlignerT5TrainStep(a, w, FusedAdamW(a, lr=1e-3))
    opt_b = FusedAdamW(b, lr=1e-3)
    for flat, start, lens, rows, l_max, flat_q, lq, Tq in batches:
        loss_a = step.step_device(flat, start, lens, rows, l_max, flat_q, lq, Tq)
        cu = ops.cu_seqlens(lens)
        x = ops.pack_varlen(flat, start, cu, rows)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = b.forward_packed(x, cu)
        loss_b = td.t5_decoder_loss(y, cu, l_max, flat_q, ops.cu_seqlens(lq), Tq, w)
        loss_b.backward()
        opt_b.step()
        opt_b.zero_grad(set_to_none=True)
        assert torch.equal(loss_a, loss_b)
    for (n, pa), pb in zip(a.named_parameters(), b.parameters()):
        assert torch.equal(pa, pb), n


def test_train_step_gradients_scale_exactly_with_the_loss_scale():
    w = _decoder_weights(D, H, 1024, NB, V, seed=22)
    batch = _batch(3)
    grads = []
    for scale in (1.0, 65536.0):
        a = _aligner(1)
        loss = td.AlignerT5TrainStep(a, w, loss_scale=scale).step_device(*batch)
        grads.append(([p.grad.clone() for p in a.parameters()], loss))
    (g1, l1), (g2, l2) = grads
    assert torch.equal(l1, l2)
    for x, y in zip(g1, g2):
        assert torch.equal(x * 65536.0, y)


def test_train_step_launch_count_and_single_gpu_scope():
    w = _decoder_weights(D, H, 1024, NB, V, seed=23)
    a = _aligner(2)
    step = td.AlignerT5TrainStep(a, w, FusedAdamW(a))
    batch = _batch(4)
    step.step_device(*batch)  # first step: also casts the four bf16 parameter copies
    n0 = _lib.launch_count
    step.step_device(*batch)
    # DESIGN section 3: 2 cu_seqlens + pack + 3 aligner forward, cast + decoder inputs, 12 per block forward, final norm + head (5) +
    # norm backward, 16 per block backward less block 0's self-attention (6), 7 aligner backward, 2 AdamW = 28 n_blocks + 18
    assert _lib.launch_count - n0 == 28 * NB + 18
    from thinkdiff_mlre_b200.optim import DeviceGradScaler

    for kw in ({"grad_scaler": DeviceGradScaler("cuda")}, {"max_grad_norm": 1.0}, {"accum_grad_iters": 2}):
        with pytest.raises(NotImplementedError, match="AlignerT5TrainStep"):
            td.AlignerT5TrainStep(a, w, FusedAdamW(a), **kw)
    a._dp = object()  # what enable_data_parallel leaves behind (it needs a process group)
    with pytest.raises(NotImplementedError, match="AlignerT5TrainStep runs on one GPU"):
        step.step_device(*batch)
    a._dp = None


# ------------------------------------------------------------------------------------------------ against HF and float64
def _hf_model(d, H, d_ff, n_blocks, V, seed):
    import transformers

    cfg = transformers.T5Config(vocab_size=V, d_model=d, d_kv=64, d_ff=d_ff, num_layers=1, num_decoder_layers=n_blocks, num_heads=H,
                                relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                                feed_forward_proj="gated-gelu", use_cache=False, layer_norm_epsilon=EPS, tie_word_embeddings=False,
                                decoder_start_token_id=0, pad_token_id=0)
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.device("cuda"):
        model = transformers.T5ForConditionalGeneration(cfg).eval()
    with torch.no_grad():
        for name, p in model.named_parameters():
            r = torch.randn(p.shape, generator=g, device="cuda")
            if p.dim() == 1:
                p.copy_(1.0 + 0.1 * r)
            elif "relative_attention_bias" in name:
                p.copy_(0.5 * r)
            elif name in ("shared.weight", "lm_head.weight"):
                p.copy_(2.0 * r * d ** -0.5)  # logits O(1); the embedding rows are renormalised by the first pre-norm
            else:  # q / k: scores O(1); the decoder's o / wo: residual stream O(1) over 3 n_blocks sublayers
                scale = 0.25 if name.endswith(("q.weight", "k.weight")) else 1.0
                if name.startswith("decoder.") and name.endswith("o.weight"):
                    scale = (3 * n_blocks) ** -0.5
                p.copy_(r * scale * p.shape[1] ** -0.5)
    return model.to(torch.bfloat16).requires_grad_(False)


def _eager_aligner(a):
    from transformers.models.t5.modeling_t5 import T5LayerNorm

    e = torch.nn.Sequential(torch.nn.Linear(a.mm_hidden_size, a.hidden_size), torch.nn.GELU(), torch.nn.Linear(a.hidden_size, a.hidden_size),
                            T5LayerNorm(a.hidden_size, EPS)).cuda()
    e.load_state_dict(a.state_dict())
    return e


@pytest.mark.parametrize("din,d,H,d_ff,n_blocks,V", [(256, 512, 8, 1056, 3, 512), (3584, 4096, 64, 10240, 2, 32128)])
def test_loss_and_aligner_gradients_closer_to_float64_than_hf(din, d, H, d_ff, n_blocks, V):
    model = _hf_model(d, H, d_ff, n_blocks, V, seed=d + n_blocks)
    w = td.T5ForDecoderWeights.from_module(model)
    torch.manual_seed(9)
    a = td.ThinkDiffAligner(din, d).cuda()
    with torch.no_grad():
        a[3].weight.copy_(1.0 + 0.1 * torch.randn(d))
    e = _eager_aligner(a)
    lens_k, lens_q = [5, 77, 1, 40], [12, 1, 33, 20]
    B, Lk = len(lens_k), max(lens_k)
    gen = torch.Generator(device="cuda").manual_seed(17)
    x = torch.randn((sum(lens_k), din), generator=gen, device="cuda").to(torch.bfloat16)
    labels = _labels(lens_q, V, seed=19)
    flat, lq, Tq = td.pack_labels(labels, V)
    start = torch.tensor([0] + lens_k[:-1], device="cuda").cumsum(0)

    loss = td.AlignerT5TrainStep(a, w).step_device(x, start, torch.tensor(lens_k, dtype=torch.int32, device="cuda"), sum(lens_k), Lk,
                                                   flat, lq.cuda(), Tq)
    ours = [p.grad for p in a.parameters()]

    cu_k = [0] + torch.tensor(lens_k).cumsum(0).tolist()
    xp = torch.zeros((B, Lk, din), dtype=torch.bfloat16, device="cuda")
    mask = torch.zeros((B, Lk), dtype=torch.long, device="cuda")
    for b, n in enumerate(lens_k):
        xp[b, :n] = x[cu_k[b] : cu_k[b + 1]]
        mask[b, :n] = 1
    with torch.autocast("cuda", dtype=torch.bfloat16):
        hf_loss = model(encoder_outputs=(e(xp),), attention_mask=mask, labels=labels).loss
    hf_loss.backward()
    hf = [p.grad for p in e.parameters()]

    a64 = _eager_aligner(a).double()
    y64 = a64(x.double())
    w64 = oref.weights_from_model(model)
    r_loss = oref.loss(y64, flat, [0] + lq.cumsum(0).tolist(), cu_k, w64)
    r_loss.backward()
    ref = [p.grad for p in a64.parameters()]

    for name, o, h, r in zip(("W1", "b1", "W2", "b2", "g"), ours, hf, ref):
        assert _rel(o, r) <= 1.25 * _rel(h, r), (name, _rel(o, r), _rel(h, r))

    # A loss is one scalar, its error one draw of the rounding noise: compare the RMS errors over nine label draws (the one above and
    # eight forward-only ones on the same aligner rows), with the 1.25x rule's floor of 1e-4 of the loss.
    errs = [(float(loss) - float(r_loss), float(hf_loss.detach()) - float(r_loss))]
    cu_k_dev = _cu(lens_k)
    with torch.no_grad():
        y64 = a64(x.double())
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = a.forward_packed(x, cu_k_dev)
            y_hf = e(xp)
        for s in range(8):
            lab = _labels(lens_q, V, seed=100 + s)
            fl, lqs, Tqs = td.pack_labels(lab, V)
            ours_s = td.t5_decoder_loss(y, cu_k_dev, Lk, fl, ops.cu_seqlens(lqs), Tqs, w)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                hf_s = model(encoder_outputs=(y_hf,), attention_mask=mask, labels=lab).loss
            r_s = oref.loss(y64, fl, [0] + lqs.cumsum(0).tolist(), cu_k, w64)
            errs.append((float(ours_s) - float(r_s), float(hf_s) - float(r_s)))
    rms = [float(torch.tensor(c).pow(2).mean().sqrt()) for c in zip(*errs)]
    assert rms[0] <= 1.25 * rms[1] + 1e-4 * abs(float(r_loss)), (rms, errs)
