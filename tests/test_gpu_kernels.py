"""-m gpu: each native kernel, called through the C ABI, against a torch fp32 reference or the
golden vectors produced by the reference.  The 16-bit kernels run in BOTH builds of the library (h16 =
float16 -> libb2e.so, bfloat16 -> libb2e_bf16.so); tolerances follow the storage type's rounding
(2^-11 resp. 2^-8 relative)."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from distllm_b200 import _native as nv

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def dev():
    if not torch.cuda.is_available():
        pytest.fail('-m gpu tests need a CUDA device')
    return torch.device('cuda:0')


@pytest.fixture(params=[torch.float16, torch.bfloat16], ids=['f16', 'bf16'])
def h16(request):
    """The 16-bit storage type = which build of the library the call lands in."""
    return request.param


def close(got, ref, h16, scale: float = 1.0):
    """assert_close with the storage type's rounding: `scale` x (3e-3 for half, 1.2e-2 for bfloat16)."""
    t = (3e-3 if h16 == torch.float16 else 1.2e-2) * scale
    torch.testing.assert_close(got, ref, rtol=t, atol=t)


GEMM_SHAPES = [(128, 256, 64), (300, 768, 768), (1000, 2304, 768), (517, 3072, 768), (517, 768, 3072),
               (200, 384, 128), (1, 768, 768), (20000, 768, 768)]


@pytest.mark.parametrize('m,n,k', GEMM_SHAPES)
@pytest.mark.parametrize('epi', [nv.EPI_BIAS, nv.EPI_BIAS_GELU, nv.EPI_BIAS_RESID])
def test_gemm_epilogues(dev, m, n, k, epi, h16):
    g = torch.Generator(device=dev).manual_seed(m * 7 + n + k + epi)
    a = (torch.randn(m, k, device=dev, generator=g) * 0.5).to(h16)
    w = (torch.randn(n, k, device=dev, generator=g) * 0.05).to(h16)
    bias = torch.randn(n, device=dev, generator=g) * 0.1
    resid = torch.randn(m, n, device=dev, generator=g).to(h16)
    out = nv.gemm_h16(a, w, bias, resid if epi == nv.EPI_BIAS_RESID else None, epi)
    ref = a.float() @ w.float().T + bias
    if epi == nv.EPI_BIAS_GELU:
        ref = torch.nn.functional.gelu(ref)
    if epi == nv.EPI_BIAS_RESID:
        ref = ref + resid.float()
    assert out.dtype == h16 and out.shape == (m, n)
    close(out.float(), ref, h16)


def test_gemm_rejects_bad_shapes(dev, h16):
    a = torch.zeros(8, 100, device=dev, dtype=h16)
    w = torch.zeros(128, 100, device=dev, dtype=h16)
    with pytest.raises(nv.NativeError, match='K=100'):
        nv.gemm_h16(a, w, torch.zeros(128, device=dev))
    with pytest.raises(nv.NativeError, match='N=100'):
        nv.gemm_h16(torch.zeros(8, 64, device=dev, dtype=h16),
                     torch.zeros(100, 64, device=dev, dtype=h16), torch.zeros(100, device=dev))


@pytest.mark.parametrize('n,epi', [
    # CTA-pair kernel (N % 256 == 0): every epilogue the trunks use, and the residual one
    (768, nv.EPI_BIAS), (1024, nv.EPI_BIAS_GELU), (768, nv.EPI_BIAS_RESID), (1536, nv.EPI_SWIGLU),
    (1536, nv.EPI_GEGLU),
    # single-CTA kernel (N % 256 == 128; the gated epilogues need N % 256 == 0)
    (384, nv.EPI_BIAS), (640, nv.EPI_BIAS_GELU), (384, nv.EPI_BIAS_RESID)])
def test_gemm_device_row_count(dev, n, epi, h16):
    """The packed trunks pass the row count on the device (t_real): rows below it must equal the plain GEMM bit for
    bit, row tiles at or beyond it must not be written."""
    from distllm_b200.embed.encoders.weights import interleave_gate_up

    m_max, k = 20000, 256
    g = torch.Generator(device=dev).manual_seed(n + epi)
    a = (torch.randn(m_max, k, device=dev, generator=g) * 0.5).to(h16)
    w = (torch.randn(n, k, device=dev, generator=g) * 0.08).to(h16)
    if epi in (nv.EPI_SWIGLU, nv.EPI_GEGLU):
        w = interleave_gate_up(w[:n // 2], w[n // 2:]).contiguous()
    bias = torch.randn(n, device=dev, generator=g) * 0.1 if epi <= nv.EPI_BIAS_RESID else None
    resid = torch.randn(m_max, n, device=dev, generator=g).to(h16) if epi == nv.EPI_BIAS_RESID else None
    want = nv.gemm_h16(a, w, bias, resid, epi)
    for m in (1, 127, 128, 129, 255, 256, 257, m_max):
        out = torch.full_like(want, SENTINEL)
        nv.debug_gemm_rows(a, w, bias, resid, epi, torch.tensor([m], dtype=torch.int32, device=dev), out)
        assert torch.equal(out[:m], want[:m]), m
        assert (out[(m + 255) // 256 * 256:] == SENTINEL).all(), f'rows past m={m} written'


@pytest.fixture(params=[None, 5, 0, 69, 64, 193], ids=['shipping', 'two-wg-poly', 'two-wg', 'four-wg-poly', 'four-wg-vote', 'four-wg-epilogue-role'])
def att_variant(request, h16):
    """Which head_dim-64 attention kernel the calls of a test reach: the library's default (variant 65: four
    softmax warpgroups, attention5.cuh), the two-warpgroup kernel of attention3.cuh (5, 0), or the other
    four-warpgroup flavours (69: polynomial exponentials, 64: vote over the bias row, 193: a fifth warpgroup takes
    the per-tile epilogue)."""
    import ctypes

    lib = nv.load(nv.storage_of(h16))
    lib.b2e_debug_set_att3_variant.argtypes = [ctypes.c_int]
    if request.param is not None:
        assert lib.b2e_debug_set_att3_variant(request.param) == 0
    yield request.param
    lib.b2e_debug_set_att3_variant(-1)   # back to B2E_ATT3 / the built-in default


def ref_attention(qkv, mask, b, s, heads, window=0):
    """fp32 reference, one sequence at a time (S = 8192 stays in the low GBs); window > 0: |i - j| <= window."""
    out = torch.empty(b, s, heads * 64, device=qkv.device)
    i = torch.arange(s, device=qkv.device)
    band = (i[:, None] - i[None, :]).abs() <= window if window else None
    for r in range(b):
        q, k, v = qkv[r * s:(r + 1) * s].float().view(s, 3, heads, 64).permute(1, 2, 0, 3)
        vis = (mask[r] != 0)[None, :] if band is None else band & (mask[r] != 0)[None, :]
        scores = (q @ k.transpose(-1, -2) / 8.0).masked_fill_(~vis, torch.finfo(torch.float32).min)
        out[r] = (torch.softmax(scores, dim=-1) @ v).permute(1, 0, 2).reshape(s, heads * 64)
        del scores
    return out.view(b * s, heads * 64)


# Rows behind the last packed sequence hold this in K and V (alternating sign), and ctx holds it there before a
# packed call: a key read past a sequence's length, or a store past its rows, changes the result visibly.  Exact in
# both 16-bit types.
SENTINEL = 24576.0


def check_packed(qkv, mask, padded_ctx, ref, rows_ok, h16, scale, *, heads, kv_heads=None, head_dim=64, window=0):
    """The problem `padded_ctx` came from, run again on the library's padding-free token layout
    (b2e_debug_pack_layout + b2e_debug_attention_packed): rows of the valid tokens must match the fp32 reference
    (where `rows_ok`) and the padded result bit for bit; rows behind them must stay untouched.  Masks the packer
    refuses (holes, left padding, empty rows) give the identity layout and the whole padded result."""
    b, s = mask.shape
    kv_heads = kv_heads or heads
    cu, ln, t_real, src = nv.debug_pack_layout(mask, storage=nv.storage_of(h16))
    t, packed = t_real.tolist()
    if not packed:
        assert t == b * s and cu.tolist() == list(range(0, b * s + 1, s)) and ln.tolist() == [s] * b
        ctx = torch.full_like(padded_ctx, float('nan'))
        nv.debug_attention_packed(qkv, mask, cu, ln, ctx, heads, kv_heads, head_dim, window)
        assert torch.equal(ctx, padded_ctx)
        return
    src = src[:t].long()
    qcols = heads * head_dim
    qkvp = qkv.clone()
    qkvp[:t] = qkv[src]
    sign = 1.0 - 2.0 * (torch.arange(qkv.shape[1] - qcols, device=qkv.device) % 2)
    qkvp[t:, qcols:] = (SENTINEL * sign).to(qkv.dtype)
    ctx = torch.full_like(padded_ctx, float('nan'))
    ctx[t:] = SENTINEL
    nv.debug_attention_packed(qkvp, mask, cu, ln, ctx, heads, kv_heads, head_dim, window)
    assert torch.isfinite(ctx[:t].float()).all()
    assert (ctx[t:] == SENTINEL).all(), 'a store landed behind the last sequence'
    ok = rows_ok[src]
    close(ctx[:t][ok].float(), ref[src][ok], h16, scale)
    if head_dim == 128:
        # Not bit for bit: the causal kernel picks its fast softmax path (one exponential in four as a polynomial)
        # per warp of 32 query rows, by a vote that also counts the rows behind the sequence's last one -- padding
        # queries in the padded layout, the next sequence's queries in the packed one (attention4.cuh,
        # `done = __all_sync(...)`).  Both paths are exact to the storage type: within half its tolerance.
        close(ctx[:t].float(), padded_ctx[src].float(), h16, 0.5)
    else:
        assert torch.equal(ctx[:t], padded_ctx[src]), 'packed and padded layouts differ'


@pytest.mark.parametrize('b,s,heads,ragged', [(2, 128, 2, False), (2, 512, 12, False), (3, 200, 12, True),
                                              (2, 512, 12, True), (4, 37, 4, True), (5, 1, 4, False),
                                              (2, 129, 4, True), (1, 384, 12, True), (2, 640, 2, False),
                                              (1, 1026, 4, True), (3, 257, 2, True),
                                              (8, 1026, 20, True), (2, 8192, 2, True)])
def test_attention_matches_reference(dev, b, s, heads, ragged, h16, att_variant):
    g = torch.Generator(device=dev).manual_seed(b * 1000 + s)
    qkv = torch.randn(b * s, 3 * heads * 64, device=dev, generator=g).to(h16)
    mask = torch.ones(b, s, dtype=torch.int64, device=dev)
    if ragged:
        for i in range(b):
            mask[i, max(1, s - 17 * (i + 1)):] = 0
    ctx = nv.attention_d64(qkv, mask, b, s, heads)
    ref = ref_attention(qkv, mask, b, s, heads)
    close(ctx.float(), ref, h16, 2.0)
    check_packed(qkv, mask, ctx, ref, mask.bool().view(-1), h16, 2.0, heads=heads)


# every edge of the 64-key chunks and 128-row query tiles, mixed in one batch
EDGE_LENGTHS = [1, 63, 64, 65, 127, 128, 129, 255, 257, 300]


@pytest.mark.parametrize('kind', ['full', 'window'])
def test_attention_packed_length_edges(dev, kind, h16, att_variant):
    """Sequences of 1 .. S tokens back to back on the packed layout: Q tiles start at arbitrary rows, the last key
    chunk of every sequence runs into the next one, partial last tiles leave row by row."""
    attention_length_edges(dev, kind, h16)


def test_attention_causal_d128_packed_length_edges(dev, h16):
    attention_length_edges(dev, 'causal', h16)


def attention_length_edges(dev, kind, h16):
    b, s = len(EDGE_LENGTHS), max(EDGE_LENGTHS)
    heads, kv_heads, d, window = (6, 6, 64, 0) if kind == 'full' else (4, 4, 64, 64) if kind == 'window' else (4, 2, 128, 100)
    g = torch.Generator(device=dev).manual_seed(17 + len(kind))
    qkv = torch.randn(b * s, (heads + 2 * kv_heads) * d, device=dev, generator=g).to(h16)
    lens = torch.tensor(EDGE_LENGTHS[3:] + EDGE_LENGTHS[:3])   # not sorted: short rows between long ones
    mask = (torch.arange(s)[None] < lens[:, None]).long().to(dev)
    if kind == 'causal':
        ctx = nv.attention_causal_d128(qkv, mask, b, s, heads, kv_heads, window)
        ref, rows_ok = ref_attention_causal(qkv, mask, b, s, heads, kv_heads, window)
    else:
        ctx = nv.attention_d64_window(qkv, mask, b, s, heads, window) if window else nv.attention_d64(qkv, mask, b, s, heads)
        ref, rows_ok = ref_attention(qkv, mask, b, s, heads, window), torch.ones(b * s, dtype=torch.bool, device=dev)
    valid = mask.bool().view(-1)
    close(ctx.float()[valid & rows_ok], ref[valid & rows_ok], h16, 2.0)
    check_packed(qkv, mask, ctx, ref, rows_ok, h16, 2.0, heads=heads, kv_heads=kv_heads, head_dim=d, window=window)


def test_attention_mask_with_holes_and_fully_masked_row(dev, h16, att_variant):
    """Arbitrary 0/1 masks (left padding, holes); an all-zero mask degenerates to a uniform
    distribution over the S keys exactly like HF's additive most-negative-finite mask."""
    b, s, heads = 3, 96, 4
    g = torch.Generator(device=dev).manual_seed(9)
    qkv = torch.randn(b * s, 3 * heads * 64, device=dev, generator=g).to(h16)
    mask = torch.ones(b, s, dtype=torch.int64, device=dev)
    mask[0, :40] = 0            # left padding
    mask[1, 10:20] = 0          # a hole
    mask[2, :] = 0              # nothing attended
    ctx = nv.attention_d64(qkv, mask, b, s, heads)
    ref = ref_attention(qkv, mask, b, s, heads)
    assert torch.isfinite(ctx.float()).all()
    close(ctx.float(), ref, h16, 2.0)
    # the packer refuses each of these rows on its own: identity layout, the padded result bit for bit
    for bad in range(b):
        m = torch.ones_like(mask)
        m[:, 60:] = 0
        m[bad] = mask[bad]
        check_packed(qkv, m, nv.attention_d64(qkv, m, b, s, heads), None, None, h16, 2.0, heads=heads)


def test_attention_many_items_per_cta(dev, h16, att_variant):
    """More work items than SMs: the persistent CTAs recycle Q buffers, ring stages and TMEM slots."""
    b, s, heads = 40, 300, 12
    g = torch.Generator(device=dev).manual_seed(77)
    qkv = torch.randn(b * s, 3 * heads * 64, device=dev, generator=g).to(h16)
    lens = torch.randint(1, s + 1, (b,), generator=torch.Generator().manual_seed(5))
    mask = (torch.arange(s)[None] < lens[:, None]).long().to(dev)
    ctx = nv.attention_d64(qkv, mask, b, s, heads)
    ref = ref_attention(qkv, mask, b, s, heads)
    valid = mask.bool().view(-1)
    close(ctx.float()[valid], ref[valid], h16, 2.0)
    assert torch.isfinite(ctx.float()).all()
    check_packed(qkv, mask, ctx, ref, valid, h16, 2.0, heads=heads)


def test_attention_large_scores_trigger_rescale(dev, h16, att_variant):
    """Scores that grow along the key axis force the lazy online-softmax rescale path."""
    b, s, heads = 2, 512, 2
    g = torch.Generator(device=dev).manual_seed(78)
    qkv = torch.randn(b * s, 3 * heads * 64, device=dev, generator=g)
    # keys later in the sequence get larger norms -> row maxima jump by far more than 2^8
    ramp = torch.linspace(0.2, 6.0, s, device=dev).repeat(b)[:, None]
    qkv[:, heads * 64:2 * heads * 64] *= ramp
    qkv = qkv.to(h16)
    mask = torch.ones(b, s, dtype=torch.int64, device=dev)
    ctx = nv.attention_d64(qkv, mask, b, s, heads)
    close(ctx.float(), ref_attention(qkv, mask, b, s, heads), h16, 3.0)
    # the same ramp on the packed layout: the first sequence stops mid-chunk, its successor starts there
    mask[0, 301:] = 0
    mask[1, 450:] = 0
    ctx = nv.attention_d64(qkv, mask, b, s, heads)
    ref = ref_attention(qkv, mask, b, s, heads)
    valid = mask.bool().view(-1)
    close(ctx.float()[valid], ref[valid], h16, 3.0)
    check_packed(qkv, mask, ctx, ref, valid, h16, 3.0, heads=heads)


@pytest.mark.parametrize('h', [256, 768, 1024, 1280])
def test_layernorm(dev, h, h16):
    g = torch.Generator(device=dev).manual_seed(h)
    x = (torch.randn(1003, h, device=dev, generator=g) * 3 + 1).to(h16)
    gamma = torch.randn(h, device=dev, generator=g)
    beta = torch.randn(h, device=dev, generator=g)
    ref = torch.nn.functional.layer_norm(x.float(), (h,), gamma, beta, 1e-12)
    torch.testing.assert_close(nv.layernorm(x, gamma, beta, 1e-12, torch.float32), ref, rtol=1e-4, atol=1e-4)
    close(nv.layernorm(x, gamma, beta, 1e-12).float(), ref, h16, 2.0)


@pytest.mark.parametrize('case', ['ragged', 'full', 'single', 'left_padded_like'])
def test_pool_mean_matches_reference_vectors(dev, pool_golden, case):
    emb = torch.from_numpy(pool_golden[f'{case}/emb']).to(dev)
    mask = torch.from_numpy(pool_golden[f'{case}/mask']).to(dev)
    got = nv.pool_mean(emb, mask)
    np.testing.assert_allclose(got.cpu().numpy(), pool_golden[f'{case}/mean'], rtol=1e-5, atol=1e-6)
    # the caller's mask is rewritten exactly like distllm/embed/poolers/mean.py:35-36
    np.testing.assert_array_equal(mask.cpu().numpy(), pool_golden[f'{case}/mask_after'])


@pytest.mark.parametrize('dtype', [torch.bfloat16, torch.float16])
def test_pool_mean_half_inputs(dev, dtype):
    from oracle import pooling as opool

    g = torch.Generator().manual_seed(4)
    emb = torch.randn(6, 50, 512, generator=g).to(dtype)
    lens = torch.tensor([50, 3, 17, 17, 1, 44])
    mask = (torch.arange(50)[None] < lens[:, None]).long()
    ref = opool.average_pool(emb.float(), mask.clone())
    got = nv.pool_mean(emb.to(dev), mask.to(dev))
    assert got.dtype == torch.float32
    torch.testing.assert_close(got.cpu(), ref, rtol=1e-2, atol=1e-2)


def test_pool_mean_per_row_mode_and_no_mutation(dev):
    g = torch.Generator().manual_seed(5)
    emb = torch.randn(4, 30, 256, generator=g)
    lens = [30, 7, 12, 2]
    mask = (torch.arange(30)[None] < torch.tensor(lens)[:, None]).long()
    ref = torch.stack([emb[i, 1:n - 1].mean(0) if n > 2 else torch.zeros(256) for i, n in enumerate(lens)])
    m = mask.to(dev)
    got = nv.pool_mean(emb.to(dev), m, nv.POOL_MEAN_PER_ROW, mutate_mask=False)
    torch.testing.assert_close(got.cpu(), ref, rtol=1e-5, atol=1e-6)
    assert torch.equal(m.cpu(), mask)


@pytest.mark.parametrize('case', ['full', 'single', 'left_padded_like', 'leftpad'])
def test_pool_last_token_matches_reference_vectors(dev, pool_golden, case):
    emb = torch.from_numpy(pool_golden[f'{case}/emb']).to(dev)
    mask = torch.from_numpy(pool_golden[f'{case}/mask']).to(dev)
    got = nv.pool_last_token(emb, mask)
    np.testing.assert_array_equal(got.cpu().numpy(), pool_golden[f'{case}/last'])


def test_adjacent_cosine_matches_reference_vectors(dev, semantic_golden):
    emb = torch.from_numpy(semantic_golden['emb']).to(dev)
    ranges = [tuple(r) for r in semantic_golden['doc_ranges']]
    doc_id = torch.empty(len(emb), dtype=torch.int32)
    for k, (lo, hi) in enumerate(ranges):
        doc_id[lo:hi] = k
    d = nv.adjacent_cosine_dist(emb, doc_id.to(dev)).cpu().numpy()
    for k, (lo, hi) in enumerate(ranges):
        np.testing.assert_allclose(d[lo:hi - 1], semantic_golden[f'dist/{k}'], rtol=0, atol=5e-7)
        if hi < len(emb):
            assert np.isnan(d[hi - 1]), 'pairs across a document boundary must be NaN'
    # no doc ids: plain consecutive distances; 0/1-row inputs: nothing to compute
    plain = nv.adjacent_cosine_dist(emb).cpu().numpy()
    assert not np.isnan(plain).any() and plain.shape == (len(emb) - 1,)
    assert nv.adjacent_cosine_dist(emb[:1]).shape == (0,)


def test_product_split_equals_oracle_split_on_same_embeddings(dev, semantic_golden):
    """Discrete output: on identical embeddings the native distance kernel + host percentile split
    must give exactly the reference's row groups."""
    from distllm_b200.embed.embedders.semantic_chunk import build_chunks
    from oracle import semantic as osem

    emb = semantic_golden['emb']
    ranges = [tuple(int(v) for v in r) for r in semantic_golden['doc_ranges']]
    dev_emb = torch.from_numpy(emb).to(dev)
    for pct in (50, 90, 95):
        got = []
        for lo, hi in ranges:
            d = nv.adjacent_cosine_dist(dev_emb[lo:hi].contiguous()).cpu().numpy().astype(np.float64)
            got.extend((lo + s, lo + e) for s, e in build_chunks(d, pct))
        assert got == osem.split_rows(emb, ranges, pct)


def test_l2_normalize(dev):
    x = torch.randn(33, 768, device=dev)
    x[5] = 0
    ref = torch.nn.functional.normalize(x, p=2, dim=-1)
    torch.testing.assert_close(nv.l2_normalize_(x.clone()), ref, rtol=1e-6, atol=1e-7)


# ---------------------------------------------------------------------------- Mistral-family kernels
@pytest.mark.parametrize('m,i,k', [(128, 128, 64), (300, 768, 512), (1000, 1792, 1024), (5, 256, 4096)])
def test_gemm_swiglu_epilogue(dev, m, i, k, h16):
    """gate/up rows interleaved in blocks of 64 -> silu(gate) * up, no bias, [M, I] out."""
    from distllm_b200.embed.encoders.weights import interleave_gate_up

    g = torch.Generator(device=dev).manual_seed(m + i + k)
    a = (torch.randn(m, k, device=dev, generator=g) * 0.5).to(h16)
    gate = (torch.randn(i, k, device=dev, generator=g) * 0.08).to(h16)
    up = (torch.randn(i, k, device=dev, generator=g) * 0.08).to(h16)
    out = nv.gemm_h16(a, interleave_gate_up(gate, up).contiguous(), None, None, nv.EPI_SWIGLU)
    ref = torch.nn.functional.silu(a.float() @ gate.float().T) * (a.float() @ up.float().T)
    assert out.dtype == h16 and out.shape == (m, i)
    close(out.float(), ref, h16, 1.3)


def test_gemm_without_bias(dev, h16):
    g = torch.Generator(device=dev).manual_seed(4)
    a = torch.randn(200, 256, device=dev, generator=g).to(h16)
    w = (torch.randn(512, 256, device=dev, generator=g) * 0.05).to(h16)
    out = nv.gemm_h16(a, w, None)
    close(out.float(), a.float() @ w.float().T, h16)


def ref_attention_causal(qkv, mask, b, s, heads, kv_heads, window):
    """fp32 reference, one sequence at a time; (context, query rows that see at least one key)."""
    d = 128
    i = torch.arange(s, device=qkv.device)[:, None]
    j = torch.arange(s, device=qkv.device)[None, :]
    causal = j <= i
    if window:
        causal = causal & (i - j < window)
    out = torch.empty(b, s, heads * d, device=qkv.device)
    alive = torch.empty(b, s, dtype=torch.bool, device=qkv.device)
    for r in range(b):
        x = qkv[r * s:(r + 1) * s].float()
        q = x[:, :heads * d].view(s, heads, d).transpose(0, 1)
        k = x[:, heads * d:(heads + kv_heads) * d].view(s, kv_heads, d).transpose(0, 1)
        v = x[:, (heads + kv_heads) * d:].view(s, kv_heads, d).transpose(0, 1)
        k = k.repeat_interleave(heads // kv_heads, dim=0)
        v = v.repeat_interleave(heads // kv_heads, dim=0)
        vis = causal & (mask[r] != 0)[None, :]
        scores = ((q @ k.transpose(-1, -2)) * d ** -0.5).masked_fill_(~vis, float('-inf'))
        p = torch.nan_to_num(torch.softmax(scores, dim=-1), nan=0.0)
        del scores
        out[r] = (p @ v).transpose(0, 1).reshape(s, heads * d)
        alive[r] = vis.any(-1)
    return out.view(b * s, heads * d), alive.view(b * s)


CAUSAL_CASES = [
    # b, s, heads, kv_heads, window, padding
    (2, 128, 2, 1, 0, 'none'), (2, 256, 4, 2, 0, 'none'), (3, 200, 4, 1, 0, 'right'),
    (2, 513, 2, 2, 0, 'right'), (2, 320, 4, 2, 80, 'right'), (2, 320, 4, 2, 80, 'left'),
    (1, 1100, 2, 1, 0, 'none'), (1, 1100, 2, 1, 300, 'left'), (4, 37, 2, 1, 16, 'right'),
    (5, 1, 2, 2, 0, 'none'), (2, 640, 8, 2, 128, 'none'), (2, 300, 4, 4, 1, 'none'),
    (2, 400, 2, 1, 64, 'right'), (2, 400, 2, 1, 65, 'left'),
    # production lengths: Mistral-7B's S = 4096 without and with its window, positions far past the window
    (2, 4096, 4, 1, 0, 'right'), (2, 4096, 2, 1, 4096, 'right'), (2, 8192, 2, 1, 4096, 'right'),
    (2, 2049, 2, 1, 1000, 'left'),
]


@pytest.mark.parametrize('b,s,heads,kv_heads,window,padding', CAUSAL_CASES)
def test_attention_causal_d128_matches_reference(dev, b, s, heads, kv_heads, window, padding, h16):
    g = torch.Generator(device=dev).manual_seed(b * 1000 + s + window)
    qkv = torch.randn(b * s, (heads + 2 * kv_heads) * 128, device=dev, generator=g).to(h16)
    mask = torch.ones(b, s, dtype=torch.int64, device=dev)
    for r in range(b):
        n_pad = min(s - 1, 23 * r + (5 if padding != 'none' else 0)) if padding != 'none' else 0
        if padding == 'right' and n_pad:
            mask[r, s - n_pad:] = 0
        if padding == 'left' and n_pad:
            mask[r, :n_pad] = 0
    ctx = nv.attention_causal_d128(qkv, mask, b, s, heads, kv_heads, window)
    ref, alive = ref_attention_causal(qkv, mask, b, s, heads, kv_heads, window)
    assert torch.isfinite(ctx.float()).all()
    # rows that see no key at all (queries inside left padding) are unspecified; everything else,
    # including padded query positions that still see attended keys, must match
    close(ctx.float()[alive], ref[alive], h16, 2.0)
    check_packed(qkv, mask, ctx, ref, alive, h16, 2.0, heads=heads, kv_heads=kv_heads, head_dim=128, window=window)


def test_attention_causal_d128_many_items_and_rescale(dev, h16):
    """More items than SMs with mixed lengths, and key norms that grow along the sequence so the lazy
    rescale path runs on top of the causal/window edge masking."""
    b, s, heads, kv_heads, window = 24, 700, 8, 2, 333
    g = torch.Generator(device=dev).manual_seed(91)
    qkv = torch.randn(b * s, (heads + 2 * kv_heads) * 128, device=dev, generator=g)
    ramp = torch.linspace(0.2, 4.0, s, device=dev).repeat(b)[:, None]
    qkv[:, heads * 128:(heads + kv_heads) * 128] *= ramp
    qkv = qkv.to(h16)
    lens = torch.randint(1, s + 1, (b,), generator=torch.Generator().manual_seed(6))
    mask = (torch.arange(s)[None] < lens[:, None]).long().to(dev)
    ctx = nv.attention_causal_d128(qkv, mask, b, s, heads, kv_heads, window)
    ref, alive = ref_attention_causal(qkv, mask, b, s, heads, kv_heads, window)
    sel = alive & mask.bool().view(-1)
    assert torch.isfinite(ctx.float()).all()
    close(ctx.float()[sel], ref[sel], h16, 3.0)
    check_packed(qkv, mask, ctx, ref, alive, h16, 3.0, heads=heads, kv_heads=kv_heads, head_dim=128, window=window)


# ---------------------------------------------------------------------------- exact inner-product top-k
def check_topk_against_oracle(queries, corpus, k, scores, idx, atol=2e-5):
    from oracle import search as osearch

    q = queries.shape[0]
    ref_s, ref_i = osearch.topk_inner_product(queries.cpu().numpy(), corpus.float().cpu().numpy(), k)
    kk = ref_s.shape[1]
    got_s, got_i = scores.cpu().numpy(), idx.cpu().numpy()
    # scores: fp32 dot products in a different summation order
    np.testing.assert_allclose(got_s[:, :kk], ref_s, rtol=0, atol=atol)
    assert (np.diff(got_s[:, :kk], axis=1) <= 0).all()
    if kk < k:   # fewer rows than k: the tail is marked empty
        assert (got_i[:, kk:] == -1).all() and np.isinf(got_s[:, kk:]).all()
    # indices: identical wherever the oracle's neighbouring scores are not within rounding of each other
    full = queries.cpu().numpy().astype(np.float64) @ corpus.float().cpu().numpy().astype(np.float64).T
    for r in range(q):
        assert len(set(got_i[r, :kk].tolist())) == kk
        np.testing.assert_allclose(full[r, got_i[r, :kk]], ref_s[r], rtol=0, atol=atol)
        clear = np.abs(np.diff(ref_s[r])) > 5 * atol
        stable = np.concatenate([[True], clear]) & np.concatenate([clear, [True]])
        assert (got_i[r, :kk][stable] == ref_i[r][stable]).all()


@pytest.mark.parametrize('q,n,h,k', [(1, 1000, 768, 10), (7, 5000, 768, 100), (16, 20000, 768, 5),
                                     (33, 3000, 256, 64), (3, 17, 128, 8), (2, 5, 768, 10),
                                     (5, 40000, 1280, 256), (4, 2000, 4096, 20), (1, 1, 768, 1)])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_topk_inner_product_matches_oracle(dev, q, n, h, k, dtype):
    from oracle import search as osearch

    g = torch.Generator(device=dev).manual_seed(q * 31 + n + k)
    if dtype == torch.bfloat16 and h % 256:
        with pytest.raises(nv.NativeError, match='multiple of 256'):
            nv.topk_ip(torch.zeros(q, h, device=dev), torch.zeros(n, h, device=dev, dtype=dtype), k)
        return
    corpus = torch.randn(n, h, device=dev, generator=g)
    corpus = corpus / corpus.norm(dim=1, keepdim=True)
    queries = torch.randn(q, h, device=dev, generator=g)
    queries = queries / queries.norm(dim=1, keepdim=True)
    corpus = corpus.to(dtype).contiguous()
    scores, idx = nv.topk_ip(queries, corpus, k)
    check_topk_against_oracle(queries, corpus, k, scores, idx)


@pytest.mark.parametrize('q,n,h,k', [(1, 40000, 768, 10), (16, 100000, 768, 100), (5, 70001, 1280, 256),
                                     (33, 50000, 256, 64), (3, 32768, 128, 1), (7, 33000, 4096, 20)])
@pytest.mark.parametrize('normalised', [True, False])
def test_topk_tensor_core_scan_matches_oracle(dev, q, n, h, k, normalised):
    """b2e_topk_ip_tc: TF32 scan on the tensor cores, exact fp32 decision -- the SAME contract as b2e_topk_ip."""
    g = torch.Generator(device=dev).manual_seed(q * 17 + n + k)
    corpus = torch.randn(n, h, device=dev, generator=g)
    queries = torch.randn(q, h, device=dev, generator=g)
    if normalised:
        corpus = corpus / corpus.norm(dim=1, keepdim=True)
        queries = queries / queries.norm(dim=1, keepdim=True)
        atol = 2e-5
    else:   # row norms spread over a factor of four: the margin is sized by the LARGEST norm
        corpus = corpus * (0.5 + 1.5 * torch.rand(n, 1, device=dev, generator=g))
        atol = 2e-5 * float(corpus.norm(dim=1).max() * queries.norm(dim=1).max())
    corpus = corpus.contiguous()
    max_norm = nv.max_row_norm(corpus)
    assert abs(max_norm - float(corpus.norm(dim=1).max())) <= 1e-5 * max_norm
    scores, idx = nv.topk_ip(queries, corpus, k, max_norm=max_norm)
    # normalised rows (what the reference indexes: faiss.normalize_L2, search.py:258-278) must stay on the fast
    # path; with spread-out norms the one global bound may be too loose and the call may redo itself exactly
    if normalised:
        assert not nv.topk_tc_fell_back()
    check_topk_against_oracle(queries, corpus, k, scores, idx, atol=atol)
    # and the two paths agree with each other far inside the oracle tolerance
    s2, i2 = nv.topk_ip(queries, corpus, k)
    assert torch.allclose(scores, s2, rtol=0, atol=atol / 4)
    same = (idx == i2).float().mean().item()
    assert same > 0.98, same


def test_topk_tensor_core_scan_falls_back_on_degenerate_corpus(dev):
    """Thousands of rows tie with the k-th best (a corpus of duplicates): the candidate buffer overflows, the call
    is redone by the exact scan on the device -- same scores as b2e_topk_ip bit for bit (WHICH of thousands of
    identical rows are named is not defined by either scan)."""
    g = torch.Generator(device=dev).manual_seed(5)
    base = torch.randn(8, 768, device=dev, generator=g)
    base = base / base.norm(dim=1, keepdim=True)
    corpus = base.repeat(6000, 1).contiguous()      # 48 000 rows, 8 distinct
    queries = torch.randn(3, 768, device=dev, generator=g)
    scores, idx = nv.topk_ip(queries, corpus, 10, max_norm=1.0)
    assert nv.topk_tc_fell_back()
    s2, i2 = nv.topk_ip(queries, corpus, 10)
    assert torch.equal(scores, s2) and torch.equal(idx % 8, i2 % 8)
    assert all(len(set(row.tolist())) == 10 for row in idx.cpu())
    best = (queries @ base.T).argmax(dim=1)
    assert torch.equal((idx[:, 0] % 8).cpu(), best.cpu())
    # a too-small norm bound can only shrink the margin, never corrupt memory; with the true bound it is exact
    corpus2 = torch.randn(40000, 768, device=dev, generator=g)
    s3, i3 = nv.topk_ip(queries, corpus2, 10, max_norm=nv.max_row_norm(corpus2))
    check_topk_against_oracle(queries, corpus2, 10, s3, i3, atol=2e-5 * 28 * float(queries.norm(dim=1).max()))


def test_topk_rejects_bad_arguments(dev):
    c = torch.zeros(10, 768, device=dev)
    qq = torch.zeros(2, 768, device=dev)
    with pytest.raises(nv.NativeError, match='k=300'):
        nv.topk_ip(qq, c, 300)
    with pytest.raises(nv.NativeError, match='H=100'):
        nv.topk_ip(torch.zeros(2, 100, device=dev), torch.zeros(10, 100, device=dev), 3)


# ---------------------------------------------------------------------------------- binary retrieval
@pytest.mark.parametrize('n,h,q,k,mult', [(5000, 768, 3, 10, 2), (20000, 1280, 9, 5, 4), (40, 256, 2, 8, 2),
                                          (3000, 64 * 3, 1, 100, 2)])
def test_ubinary_search_matches_oracle(n, h, q, k, mult):
    """b2e_pack_ubinary / b2e_search_ubinary vs the CPU restatement of packbits + IndexBinaryFlat + rescoring
    (oracle/search.py): packed bits and result indices bit-exact (integer / index work), scores to fp32 rounding."""
    from oracle import search as osearch

    rng = np.random.default_rng(n + h)
    corpus = rng.standard_normal((n, h)).astype(np.float32)
    corpus[rng.integers(0, n, 50)] = 0.0          # zero rows pack to all-zero bits
    if n > 100:
        corpus[100:110] = corpus[7]                # exact duplicates: Hamming ties resolved by row id
    queries = rng.standard_normal((q, h)).astype(np.float32)
    queries[0] = corpus[7] + 0.05 * rng.standard_normal(h).astype(np.float32)
    bits = nv.pack_ubinary(torch.from_numpy(corpus).cuda())
    ref_bits = osearch.quantize_ubinary(corpus)
    assert np.array_equal(bits.cpu().numpy(), ref_bits)
    scores, indices = nv.search_ubinary(torch.from_numpy(queries).cuda(), bits, k, mult)
    ref_s, ref_i = osearch.search_ubinary(queries, ref_bits, k, mult)
    kk = ref_i.shape[1]
    got_i, got_s = indices.cpu().numpy(), scores.cpu().numpy()
    # rescored scores are sums of up to h floats: order of summation differs -> compare with a tolerance, and
    # indices wherever the reference scores are not tied within that tolerance
    np.testing.assert_allclose(got_s[:, :kk], ref_s, rtol=1e-5, atol=1e-4)
    for r in range(q):
        gap = np.abs(np.diff(ref_s[r])) > 1e-3
        stable = np.concatenate(([True], gap)) & np.concatenate((gap, [True]))
        assert np.array_equal(got_i[r, :kk][stable], ref_i[r][stable]), (r, got_i[r], ref_i[r])
        assert set(got_i[r, :kk]) == set(ref_i[r])
    if kk < k:
        assert (got_i[:, kk:] == -1).all() and np.isinf(got_s[:, kk:]).all()


def test_exact_index_ubinary_through_the_retriever_surface():
    from distllm_b200.rag.search import ExactIndex
    from distllm_b200.rag.search import ExactIndexConfig
    from oracle import search as osearch

    rng = np.random.default_rng(9)
    corpus = rng.standard_normal((4000, 768)).astype(np.float32)
    index = ExactIndex(corpus, config=ExactIndexConfig(precision='ubinary', rescore_multiplier=3))
    assert index.corpus.dtype == torch.uint8 and index.corpus.shape == (4000, 96) and len(index) == 4000
    q = ExactIndex.transform(corpus[[5, 77]] + 0.1 * rng.standard_normal((2, 768)).astype(np.float32))
    res = index.search(q, top_k=4)
    ref_s, ref_i = osearch.search_ubinary(q, osearch.quantize_ubinary(corpus), 4, 3)
    assert [r[0] for r in res.total_indices] == [5, 77]
    assert res.total_indices == ref_i.tolist()
    np.testing.assert_allclose(np.array(res.total_scores), ref_s, rtol=1e-5, atol=1e-4)
    kept = index.search(q, top_k=4, score_threshold=float(ref_s[0, 1]))
    assert kept.total_indices[0] == ref_i[0, :2].tolist()


@pytest.mark.parametrize('m,i,k', [(300, 1152, 768), (1000, 2688, 1024)])
def test_gemm_geglu_epilogue(dev, m, i, k, h16):
    """ModernBERT's gated MLP: Wi rows = input | gate (transformers/models/modernbert/modeling_modernbert.py
    :88-91), interleaved in blocks of 64 for the epilogue: out = gelu(x Wi_in^T) * (x Wi_gate^T)."""
    from distllm_b200.embed.encoders.weights import interleave_gate_up

    g = torch.Generator(device=dev).manual_seed(m + i)
    a = (torch.randn(m, k, device=dev, generator=g) * 0.5).to(h16)
    w_in = (torch.randn(i, k, device=dev, generator=g) * 0.08).to(h16)
    w_gate = (torch.randn(i, k, device=dev, generator=g) * 0.08).to(h16)
    out = nv.gemm_h16(a, interleave_gate_up(w_in, w_gate).contiguous(), None, None, nv.EPI_GEGLU)
    ref = torch.nn.functional.gelu(a.float() @ w_in.float().T) * (a.float() @ w_gate.float().T)
    assert out.dtype == h16 and out.shape == (m, i)
    close(out.float(), ref, h16, 1.3)


@pytest.mark.parametrize('b,s,heads,window', [(2, 512, 4, 64), (3, 333, 2, 64), (1, 1500, 2, 64), (2, 200, 4, 16),
                                              (2, 700, 2, 300), (2, 8192, 2, 64)])
def test_attention_d64_sliding_window(dev, b, s, heads, window, h16, att_variant):
    """Bidirectional sliding window |i - j| <= window (ModernBERT's local layers) on ragged batches; rows of
    padding tiles must stay finite."""
    g = torch.Generator(device=dev).manual_seed(b * 100 + s + window)
    qkv = torch.randn(b * s, 3 * heads * 64, device=dev, generator=g).to(h16)
    mask = torch.ones(b, s, dtype=torch.int64, device=dev)
    for r in range(1, b):
        mask[r, max(1, s - 90 * r):] = 0
    ctx = nv.attention_d64_window(qkv, mask, b, s, heads, window)
    ref = ref_attention(qkv, mask, b, s, heads, window)
    valid = mask.bool().view(-1)
    assert torch.isfinite(ctx.float()).all()
    close(ctx.float()[valid], ref[valid], h16, 2.0)
    check_packed(qkv, mask, ctx, ref, valid, h16, 2.0, heads=heads, window=window)


# ------------------------------------------------------------------------- profiling instantiations
def test_profiling_instantiations_write_timelines_and_change_no_result(dev):
    """The clock64 timelines live in separate instantiations (attention: variant bit 8; pair GEMM: selected while a
    clock buffer is set): they must fill their buffers and give the production kernels' results bit for bit."""
    import ctypes

    lib = nv.load('bf16')
    lib.b2e_debug_set_att3_variant.argtypes = [ctypes.c_int]
    lib.b2e_debug_set_att3_clock.argtypes = [ctypes.c_void_p]
    lib.b2e_debug_set_clock_buffer.argtypes = [ctypes.c_void_p]
    g = torch.Generator(device=dev).manual_seed(11)
    b, s, heads = 6, 512, 4
    qkv = torch.randn(b * s, 3 * heads * 64, device=dev, generator=g).to(torch.bfloat16)
    mask = torch.ones(b, s, dtype=torch.int64, device=dev)
    try:
        for plain, timed in ((65, 321), (5, 261)):
            lib.b2e_debug_set_att3_variant(plain)
            want = nv.attention_d64(qkv, mask, b, s, heads).clone()
            buf = torch.zeros(4 * 512, dtype=torch.int64, device=dev)
            assert lib.b2e_debug_set_att3_clock(buf.data_ptr()) == 0
            nv.attention_d64(qkv, mask, b, s, heads)          # production kernel: no stamps even with a buffer set
            torch.cuda.synchronize()
            assert int((buf != 0).sum()) == 0
            lib.b2e_debug_set_att3_variant(timed)
            got = nv.attention_d64(qkv, mask, b, s, heads).clone()
            torch.cuda.synchronize()
            assert lib.b2e_debug_set_att3_clock(None) == 0
            assert torch.equal(got, want)
            assert int((buf.view(4, 2, 256)[0, 0] != 0).sum()) > 8   # the first softmax role recorded its chunks
    finally:
        lib.b2e_debug_set_att3_clock(None)
        lib.b2e_debug_set_att3_variant(-1)
    # pair GEMM
    a = (torch.randn(4096, 768, device=dev, generator=g) * 0.5).to(torch.bfloat16)
    w = (torch.randn(768, 768, device=dev, generator=g) * 0.05).to(torch.bfloat16)
    bias = torch.randn(768, device=dev, generator=g)
    want = nv.gemm_h16(a, w, bias).clone()
    buf = torch.zeros(4 * 256, dtype=torch.int64, device=dev)
    try:
        assert lib.b2e_debug_set_clock_buffer(buf.data_ptr()) == 0
        got = nv.gemm_h16(a, w, bias).clone()
        torch.cuda.synchronize()
    finally:
        assert lib.b2e_debug_set_clock_buffer(None) == 0
    assert torch.equal(got, want) and int((buf != 0).sum()) > 8
    buf.zero_()
    nv.gemm_h16(a, w, bias)
    torch.cuda.synchronize()
    assert int((buf != 0).sum()) == 0
