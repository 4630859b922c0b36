"""CPU side of the T5 attention kernels (SURVEY section 8 f-1): the fp32 reference ``tests/_t5_attention_ref.attention_packed`` the GPU
tests compare against, pinned live to transformers' ``T5Attention`` on the zero-padded batch + mask (outputs, and the gradients into
q / k / v on valid rows; pad rows get none); the per-distance relative position bias table against ``compute_bias``; and the
workspace size function."""
import pytest
import torch

import _t5_attention_ref as ref
from oracle.t5_decoder_ref import relative_position_bucket
from thinkdiff_mlre_b200 import _lib
from thinkdiff_mlre_b200.t5 import t5_position_bias_by_distance

transformers = pytest.importorskip("transformers")
H, DKV = 4, 16


def _config():
    from transformers import T5Config

    return T5Config(vocab_size=16, d_model=H * DKV, d_kv=DKV, d_ff=32, num_layers=1, num_heads=H, relative_attention_num_buckets=32,
                    relative_attention_max_distance=128, dropout_rate=0.0, is_decoder=True, use_cache=False)


class _Const(torch.nn.Module):
    """Stands in for a projection so that HF's attention core reads given q / k / v (and autograd reaches them)."""

    def __init__(self, t):
        super().__init__()
        self.t = t

    def forward(self, x):
        return self.t


def _hf_core(q_pad, k_pad, v_pad, mask, relative_bias_table=None):
    from transformers.models.t5.modeling_t5 import T5Attention

    att = T5Attention(_config(), has_relative_attention_bias=relative_bias_table is not None, layer_idx=0).eval()
    if relative_bias_table is not None:
        with torch.no_grad():
            att.relative_attention_bias.weight.copy_(relative_bias_table)
    att.q, att.k, att.v, att.o = _Const(q_pad), _Const(k_pad), _Const(v_pad), torch.nn.Identity()
    hidden = torch.zeros(q_pad.shape)
    return att(hidden, mask=mask, key_value_states=None if relative_bias_table is not None else torch.zeros(k_pad.shape))[0]


def _pad(x, cu, L):
    out = torch.zeros((len(cu) - 1, L, x.shape[1]))
    for b in range(len(cu) - 1):
        out[b, : cu[b + 1] - cu[b]] = x[cu[b] : cu[b + 1]]
    return out


def _cu(lens):
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    return cu


@pytest.mark.parametrize("lens_q,lens_k", [([5, 1, 9], [7, 3, 12]), ([1], [1]), ([12, 4], [2, 20])])
def test_attention_packed_cross_equals_hf_t5_attention_on_the_padded_batch(lens_q, lens_k):
    g = torch.Generator().manual_seed(sum(lens_k))
    cu_q, cu_k = _cu(lens_q), _cu(lens_k)
    q = torch.randn((cu_q[-1], H * DKV), generator=g, requires_grad=True)
    k = torch.randn((cu_k[-1], H * DKV), generator=g, requires_grad=True)
    v = torch.randn((cu_k[-1], H * DKV), generator=g, requires_grad=True)
    T, L = max(lens_q), max(lens_k)
    qp, kp, vp = (_pad(x.detach(), c, n).requires_grad_(True) for x, c, n in ((q, cu_q, T), (k, cu_k, L), (v, cu_k, L)))
    mask = torch.zeros((len(lens_q), 1, 1, L))
    for b, n in enumerate(lens_k):
        mask[b, ..., n:] = torch.finfo(torch.float32).min  # the encoder mask as HF's T5Stack extends it
    want = _hf_core(qp, kp, vp, mask)
    got = ref.attention_packed(q, k, v, cu_q, cu_k, H)
    up = torch.randn(want.shape, generator=g)
    for b, n in enumerate(lens_q):
        up[b, n:] = 0  # pad query rows carry no upstream gradient
        torch.testing.assert_close(got[cu_q[b] : cu_q[b + 1]], want[b, :n], rtol=1e-5, atol=1e-5)
    want.backward(up)
    got.backward(torch.cat([up[b, :n] for b, n in enumerate(lens_q)]))
    for b in range(len(lens_q)):
        torch.testing.assert_close(q.grad[cu_q[b] : cu_q[b + 1]], qp.grad[b, : lens_q[b]], rtol=1e-4, atol=1e-5)
        for x, xp in ((k, kp), (v, vp)):
            torch.testing.assert_close(x.grad[cu_k[b] : cu_k[b + 1]], xp.grad[b, : lens_k[b]], rtol=1e-4, atol=1e-5)
            assert not xp.grad[b, lens_k[b] :].any()  # masked keys: exactly no gradient


@pytest.mark.parametrize("lens", [[5, 1, 9], [40], [3, 130]])
def test_attention_packed_causal_self_with_relative_bias_equals_hf(lens):
    g = torch.Generator().manual_seed(len(lens))
    cu = _cu(lens)
    q, k, v = (torch.randn((cu[-1], H * DKV), generator=g, requires_grad=True) for _ in range(3))
    table = torch.randn((32, H), generator=g) * 0.5
    T = max(lens)
    qp, kp, vp = (_pad(x.detach(), cu, T).requires_grad_(True) for x in (q, k, v))
    causal = torch.full((T, T), torch.finfo(torch.float32).min).triu(1)[None, None].expand(len(lens), 1, T, T)
    want = _hf_core(qp, kp, vp, causal, relative_bias_table=table)
    got = ref.attention_packed(q, k, v, cu, None, H, bias_by_distance=t5_position_bias_by_distance(table))
    up = torch.randn(want.shape, generator=g)
    for b, n in enumerate(lens):
        up[b, n:] = 0
        torch.testing.assert_close(got[cu[b] : cu[b + 1]], want[b, :n], rtol=1e-5, atol=1e-5)
    want.backward(up)
    got.backward(torch.cat([up[b, :n] for b, n in enumerate(lens)]))
    for b, n in enumerate(lens):
        for x, xp in ((q, qp), (k, kp), (v, vp)):
            torch.testing.assert_close(x.grad[cu[b] : cu[b + 1]], xp.grad[b, :n], rtol=1e-4, atol=1e-5)
            assert not xp.grad[b, n:].any()  # pad rows: exactly no gradient


def test_attention_packed_sample_without_keys_gives_zeros_and_minus_inf_lse():
    q = torch.randn((3, H * DKV))
    k = torch.randn((2, H * DKV))
    o, lse = ref.attention_packed(q, k, k, [0, 2, 3], [0, 0, 2], H, return_lse=True)
    assert torch.equal(o[:2], torch.zeros((2, H * DKV))) and bool(torch.isneginf(lse[:, :2]).all())
    assert bool(torch.isfinite(lse[:, 2]).all())


def test_position_bias_by_distance_with_the_clamp_equals_hf_compute_bias():
    """The kernel reads entry min(i - j, n_dist - 1) of a [H, max_distance] table: equal to HF's bucketed bias for every
    (i >= j) pair up to T = 2000."""
    from transformers.models.t5.modeling_t5 import T5Attention

    att = T5Attention(_config(), has_relative_attention_bias=True, layer_idx=0)
    with torch.no_grad():
        att.relative_attention_bias.weight.copy_(torch.randn((32, H)))
    tab = t5_position_bias_by_distance(att.relative_attention_bias.weight)
    assert tab.shape == (H, 128) and tab.dtype == torch.float32
    T = 2000
    want = att.compute_bias(T, T)[0].detach()  # [H, T, T]
    n = torch.arange(T)[:, None] - torch.arange(T)[None, :]
    keep = n >= 0
    got = tab[:, n.clamp(0, 127)]
    assert torch.equal(got[:, keep], want[:, keep])
    # bf16 tables (the checkpoint's dtype) come out as the fp32 values of the bf16 entries
    tb = att.relative_attention_bias.weight.detach().to(torch.bfloat16)
    assert torch.equal(t5_position_bias_by_distance(tb), tb.float()[relative_position_bucket(-torch.arange(128), 32, 128)].t())


def test_attention_workspace_size_is_pure_and_monotone():
    lib = _lib.lib()
    prev = 0
    for mq in (0, 1, 127, 128, 8192, 65536):
        for h in (1, 4, 64):
            w = lib.td_t5_attention_workspace_bytes(mq, h)
            assert w > 0 and w % 256 == 0 and w >= 4 * mq * h
            assert w == lib.td_t5_attention_workspace_bytes(mq, h)
        assert lib.td_t5_attention_workspace_bytes(mq, 64) >= prev
        prev = lib.td_t5_attention_workspace_bytes(mq, 64)
