"""-m gpu: the padding-free ("packed") token layout of the pooled forward pass (csrc/pack.cuh).

The layout kernels against a Python restatement; pooled outputs that must not depend on what a handle ran before
(packed passes read rows behind the last attended token that they never write); and the packed and padded paths of
every family at production sequence lengths against the fp32 oracles."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from distllm_b200 import _native as nv
from oracle import pooling as opool

from conftest import cosine_rows

pytestmark = pytest.mark.gpu

COS_TOL = 1e-3


@pytest.fixture(scope='module')
def dev():
    if not torch.cuda.is_available():
        pytest.fail('-m gpu tests need a CUDA device')
    return torch.device('cuda:0')


def right_padded(lens, s):
    return (torch.arange(s)[None] < torch.as_tensor(lens)[:, None]).long()


def expected_layout(mask: torch.Tensor, enable: bool):
    """(cu, len, T', packed, tok_src[:T']) of pack.cuh, restated: packed iff enabled and every row is 1..1 0..0 with
    at least one 1; otherwise the identity layout (every row S long at b*S)."""
    b, s = mask.shape
    on = mask != 0
    lens = on.sum(1)
    prefix = bool((lens > 0).all() and (on == (torch.arange(s)[None] < lens[:, None])).all())
    packed = enable and prefix
    ln = lens if packed else torch.full((b,), s)
    cu = torch.cat([torch.zeros(1, dtype=torch.int64), ln.cumsum(0)])
    src = torch.cat([r * s + torch.arange(int(n)) for r, n in enumerate(ln)])
    return cu, ln, int(cu[-1]), int(packed), src


def layout_cases():
    g = torch.Generator().manual_seed(3)
    mixed = right_padded([300, 1, 64, 129, 257, 63], 300)
    holes = mixed.clone()
    holes[3, 10] = 0
    left = mixed.clone()
    left[2] = left[2].flip(0)
    empty = mixed.clone()
    empty[4] = 0
    return {
        'ragged': (mixed, True),
        'full': (torch.ones(4, 128, dtype=torch.int64), True),
        'single': (right_padded([50], 77), True),
        'b300': (right_padded(torch.randint(1, 201, (300,), generator=g), 200), True),
        's8192': (right_padded([8192, 4097, 1], 8192), True),
        'holes': (holes, True),
        'left_padding': (left, True),
        'empty_row': (empty, True),
        'disabled': (mixed, False),
    }


@pytest.mark.parametrize('case', list(layout_cases()))
def test_pack_layout_kernels(dev, case):
    mask, enable = layout_cases()[case]
    cu, ln, t_real, src = nv.debug_pack_layout(mask.to(dev), enable)
    want_cu, want_len, t, packed, want_src = expected_layout(mask, enable)
    assert t_real.tolist() == [t, packed]
    if case in ('holes', 'left_padding', 'empty_row', 'disabled'):
        assert packed == 0
    assert cu.tolist() == want_cu.tolist()
    assert ln.tolist() == want_len.tolist()
    src = src.cpu()
    assert torch.equal(src[:t].long(), want_src)
    assert (src[t:] == -1).all(), 'tok_src written past T\''


# ---------------------------------------------------------------------------- history independence
def family_model(family, request):
    from distllm_b200.embed.encoders import native as N

    if family == 'mistral':
        from conftest import tiny_mistral_variant

        return N.NativeMistralEncoder, tiny_mistral_variant('window')
    fixture, cls = {'bert': ('tiny_bert', N.NativeBertEncoder), 'esm': ('tiny_esm', N.NativeEsm2Encoder),
                    'modernbert': ('tiny_modernbert', N.NativeModernBertEncoder)}[family]
    return cls, request.getfixturevalue(fixture)


@pytest.mark.parametrize('family', ['bert', 'esm', 'modernbert', 'mistral'])
def test_pooled_output_does_not_depend_on_handle_history(dev, family, request):
    """Packed passes read rows behind the last attended token (partial GEMM tiles, the last key chunk) that they never
    write: what an earlier, larger batch left there must not reach the pooled output, bit for bit."""
    cls, (cfg, sd) = family_model(family, request)
    s = min(cfg.max_position_embeddings, 160)
    lens = [s, s // 2 + 3, s - 27]                      # the last one is not a multiple of 64
    assert lens[-1] % 64
    g = torch.Generator().manual_seed(11)
    ids = torch.randint(4, 24, (3, s), generator=g)
    mask = right_padded(lens, s)
    big_ids = torch.randint(4, 24, (9, s), generator=g)
    big_mask = torch.ones(9, s, dtype=torch.int64)
    kinds = (nv.POOL_MEAN_REF, nv.POOL_LAST_TOKEN)

    fresh = cls(cfg, sd)
    try:
        want = [fresh.encode_pooled(ids, mask, None, k, False).clone() for k in kinds]
    finally:
        fresh.close()
    used = cls(cfg, sd)
    try:
        used.encode(big_ids, big_mask)
        used.encode_pooled(big_ids, big_mask, None, nv.POOL_MEAN_REF, False)
        got = [used.encode_pooled(ids, mask, None, k, False).clone() for k in kinds]
    finally:
        used.close()
    for k, a, b in zip(kinds, want, got):
        assert torch.isfinite(a).all()
        assert torch.equal(a, b), (family, k)


# ---------------------------------------------------------------------------- production sequence lengths
def oracle_per_row(forward, sd, cfg, ids, mask):
    """The oracle one sequence at a time: its [B, heads, S, S] scores at S = 8192 would need twice the host memory."""
    return torch.cat([forward(sd, cfg, ids[r:r + 1], mask[r:r + 1]) for r in range(ids.shape[0])])


def check_cos(got, ref, what):
    cos = cosine_rows(got, ref)
    print(f'{what}: worst cosine {cos.min():.8f}')
    assert cos.min() > 1 - COS_TOL, (what, cos.min())


@pytest.mark.parametrize('theta', [1e4, 1e6])
def test_mistral_s8192_window_vs_oracle(theta):
    """Mistral-7B-v0.1's regime on a 2-layer model: head_dim 128, grouped-query attention, sliding window 4096,
    positions up to 8191 (rotary far beyond 1023); one row longer than the window, one of length 5000 (not a
    multiple of 64).  Pooled (packed layout) and per token (padded layout) against the fp32 oracle."""
    from transformers import MistralConfig

    from distllm_b200.embed.encoders.native import NativeMistralEncoder
    from distllm_b200.embed.encoders.weights import random_mistral_state_dict
    from oracle import mistral as omis

    cfg = MistralConfig(vocab_size=1000, hidden_size=256, num_hidden_layers=2, num_attention_heads=2,
                        num_key_value_heads=1, head_dim=128, intermediate_size=512, max_position_embeddings=8192,
                        rms_norm_eps=1e-5, sliding_window=4096, rope_theta=theta, initializer_range=0.02)
    assert omis.rope_theta_of(cfg) == theta
    sd = random_mistral_state_dict(cfg, seed=21, device='cpu')
    s = 8192
    ids = torch.randint(3, 1000, (2, s), generator=torch.Generator().manual_seed(22))
    mask = right_padded([s, 5000], s)
    ref_hidden = oracle_per_row(omis.mistral_forward, sd, cfg, ids, mask)
    native = NativeMistralEncoder(cfg, sd)
    try:
        got = native.encode_pooled(ids, mask, None, nv.POOL_LAST_TOKEN, False).cpu().numpy()
        check_cos(got, opool.last_token_pool(ref_hidden, mask).numpy(), f'mistral theta={theta:g} last-token')
        got = native.encode_pooled(ids, mask, None, nv.POOL_MEAN_REF, False).cpu().numpy()
        check_cos(got, opool.average_pool(ref_hidden, mask.clone()).numpy(), f'mistral theta={theta:g} mean')
        hidden = native.encode(ids, mask).cpu().numpy()
        valid = mask.bool().numpy()
        assert np.isfinite(hidden).all()
        check_cos(hidden[valid], ref_hidden.numpy()[valid], f'mistral theta={theta:g} per token')
    finally:
        native.close()


def test_modernbert_s8192_vs_oracle():
    """ModernBERT at its 8192 positions: one global and two local (|i - j| <= 64) layers, ragged; pooled (packed
    layout) and per token (padded layout) against the fp32 oracle."""
    from transformers import ModernBertConfig

    from distllm_b200.embed.encoders.native import NativeModernBertEncoder
    from distllm_b200.embed.encoders.weights import random_modernbert_state_dict
    from oracle import modernbert as omb

    cfg = ModernBertConfig(vocab_size=320, hidden_size=256, num_hidden_layers=3, num_attention_heads=4,
                           intermediate_size=384, max_position_embeddings=8192, local_attention=128,
                           global_attn_every_n_layers=3, norm_eps=1e-5, pad_token_id=0, bos_token_id=1,
                           eos_token_id=2, cls_token_id=1, sep_token_id=2, initializer_range=0.05)
    assert [omb.layer_is_global(cfg, i) for i in range(3)] == [True, False, False]
    sd = random_modernbert_state_dict(cfg, seed=23, device='cpu')
    s = 8192
    ids = torch.randint(4, 320, (2, s), generator=torch.Generator().manual_seed(24))
    mask = right_padded([s, 6001], s)
    ref_hidden = oracle_per_row(omb.modernbert_forward, sd, cfg, ids, mask)
    native = NativeModernBertEncoder(cfg, sd)
    try:
        got = native.encode_pooled(ids, mask, None, nv.POOL_MEAN_REF, False).cpu().numpy()
        check_cos(got, opool.average_pool(ref_hidden, mask.clone()).numpy(), 'modernbert mean')
        got = native.encode_pooled(ids, mask, None, nv.POOL_LAST_TOKEN, False).cpu().numpy()
        check_cos(got, opool.last_token_pool(ref_hidden, mask).numpy(), 'modernbert last-token')
        hidden = native.encode(ids, mask).cpu().numpy()
        valid = mask.bool().numpy()
        assert np.isfinite(hidden).all()
        check_cos(hidden[valid], ref_hidden.numpy()[valid], 'modernbert per token')
    finally:
        native.close()
