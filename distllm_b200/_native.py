"""ctypes binding of libb2e.so (the C ABI declared in include/b2e.h).

There is deliberately no fallback: if the library is missing, or a compute call is made without an
sm_100 device, a ``NativeError`` is raised.  Tensors cross the boundary as ``data_ptr()`` integers
plus sizes; the current torch CUDA stream is passed explicitly.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

import torch

# Two builds of the same sources (distllm_b200/build.py): they differ only in the 16-bit storage type of
# weights and activations.  libb2e.so = IEEE half, libb2e_bf16.so = bfloat16 (b2e_storage_dtype()).
LIB_PATH = Path(__file__).resolve().parent / 'libb2e.so'
LIB_PATHS = {'f16': LIB_PATH, 'bf16': LIB_PATH.with_name('libb2e_bf16.so')}
STORAGE_TORCH_DTYPE = {'f16': torch.float16, 'bf16': torch.bfloat16}
# Which build an encoder family runs on.  Measured (profiles/r02_drift_report_*.md, r02_notes.md section 1): with
# bfloat16 the 12-layer BERT and 33-layer ESM-2 shapes stay within 5e-5 cosine of the fp32 reference and the
# GEMMs sustain ~5 % more TFLOP/s under the board's power cap; the 32-layer Mistral-7B shape needs half (3.3e-5
# against 1.6e-3 with bfloat16; tolerance 1e-3).  B2E_STORAGE=f16|bf16 overrides for every family.
_STORAGE_BY_ARCH = {'bert': 'bf16', 'esm': 'bf16', 'modernbert': 'bf16', 'mistral': 'f16'}


def storage_for_arch(arch: str) -> str:
    import os

    forced = os.environ.get('B2E_STORAGE')
    if forced:
        if forced not in LIB_PATHS:
            raise NativeError(f'B2E_STORAGE={forced!r}: expected one of {sorted(LIB_PATHS)}')
        return forced
    return _STORAGE_BY_ARCH[arch]


def storage_of(dtype: torch.dtype) -> str:
    """The build whose storage type is ``dtype`` (operands of the building-block entry points)."""
    for name, dt in STORAGE_TORCH_DTYPE.items():
        if dt == dtype:
            return name
    raise NativeError(f'no libb2e build stores {dtype}: expected float16 or bfloat16 operands')

ARCH_BERT, ARCH_ESM2, ARCH_MISTRAL, ARCH_MODERNBERT = 0, 1, 2, 3
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
POOL_MEAN_REF, POOL_MEAN_PER_ROW, POOL_LAST_TOKEN = 0, 1, 2
EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RESID, EPI_SWIGLU, EPI_GEGLU = 0, 1, 2, 3, 4

_DTYPE_CODES = {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.float16: DTYPE_F16}

# every symbol include/b2e.h declares (checked by the CPU test-suite)
EXPORTS = (
    'b2e_version',
    'b2e_storage_dtype',
    'b2e_last_error',
    'b2e_num_weights',
    'b2e_check_model',
    'b2e_encoder_create',
    'b2e_encoder_destroy',
    'b2e_workspace_bytes',
    'b2e_encode',
    'b2e_encode_pooled',
    'b2e_embed_host',
    'b2e_pool_mean',
    'b2e_pool_last_token',
    'b2e_l2_normalize',
    'b2e_adjacent_cosine_dist',
    'b2e_gemm_h16',
    'b2e_attention_d64',
    'b2e_attention_d64_window',
    'b2e_attention_causal_d128',
    'b2e_topk_ip',
    'b2e_topk_ip_tc',
    'b2e_max_row_norm',
    'b2e_pack_ubinary',
    'b2e_search_ubinary',
    'b2e_layernorm',
)
# profiling and test hooks declared in include/b2e_debug.h (tools/ and tests/ only; the package never calls them)
DEBUG_EXPORTS = (
    'b2e_debug_set_att3_clock',
    'b2e_debug_set_att3_flags',
    'b2e_debug_set_pair_flags',
    'b2e_debug_set_clock_buffer',
    'b2e_debug_set_layers',
    'b2e_debug_set_att3_variant',
    'b2e_debug_set_packing',
    'b2e_debug_topk_tc_fell_back',
    'b2e_debug_pack_layout',
    'b2e_debug_gemm_rows',
    'b2e_debug_attention_packed',
)


class NativeError(RuntimeError):
    """Raised when libb2e.so is missing or a native call fails."""


class ModelDesc(C.Structure):
    """Mirror of ``B2EModelDesc``."""

    _fields_ = [
        ('arch', C.c_int32),
        ('num_layers', C.c_int32),
        ('hidden', C.c_int32),
        ('heads', C.c_int32),
        ('kv_heads', C.c_int32),
        ('head_dim', C.c_int32),
        ('intermediate', C.c_int32),
        ('vocab', C.c_int32),
        ('max_pos', C.c_int32),
        ('type_vocab', C.c_int32),
        ('eps', C.c_float),
        ('rope_theta', C.c_float),
        ('sliding_window', C.c_int32),
        ('reserved', C.c_int32),
        ('rope_theta_local', C.c_float),
        ('global_every', C.c_int32),
    ]


_libs: dict[str, C.CDLL] = {}


def _declare(lib: C.CDLL) -> None:
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.b2e_version.restype = i32
    lib.b2e_version.argtypes = []
    lib.b2e_storage_dtype.restype = i32
    lib.b2e_storage_dtype.argtypes = []
    lib.b2e_last_error.restype = C.c_char_p
    lib.b2e_last_error.argtypes = []
    lib.b2e_num_weights.restype = i32
    lib.b2e_num_weights.argtypes = [C.POINTER(ModelDesc)]
    lib.b2e_check_model.restype = i32
    lib.b2e_check_model.argtypes = [C.POINTER(ModelDesc)]
    lib.b2e_encoder_create.restype = i32
    lib.b2e_encoder_create.argtypes = [C.POINTER(ModelDesc), C.POINTER(vp), i32, i32, C.POINTER(vp)]
    lib.b2e_encoder_destroy.restype = None
    lib.b2e_encoder_destroy.argtypes = [vp]
    lib.b2e_workspace_bytes.restype = i64
    lib.b2e_workspace_bytes.argtypes = [vp, i32, i32]
    lib.b2e_encode.restype = i32
    lib.b2e_encode.argtypes = [vp, vp, vp, vp, i32, i32, vp, i32, vp]
    lib.b2e_encode_pooled.restype = i32
    lib.b2e_encode_pooled.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]
    lib.b2e_embed_host.restype = i32
    lib.b2e_embed_host.argtypes = [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]
    lib.b2e_pool_mean.restype = i32
    lib.b2e_pool_mean.argtypes = [vp, i32, vp, i32, i32, i32, i32, i32, vp, vp]
    lib.b2e_pool_last_token.restype = i32
    lib.b2e_pool_last_token.argtypes = [vp, i32, vp, i32, i32, i32, vp, vp]
    lib.b2e_l2_normalize.restype = i32
    lib.b2e_l2_normalize.argtypes = [vp, i64, i32, vp]
    lib.b2e_adjacent_cosine_dist.restype = i32
    lib.b2e_adjacent_cosine_dist.argtypes = [vp, i32, i64, i32, vp, vp, vp]
    lib.b2e_gemm_h16.restype = i32
    lib.b2e_gemm_h16.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.b2e_attention_d64.restype = i32
    lib.b2e_attention_d64.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.b2e_attention_d64_window.restype = i32
    lib.b2e_attention_d64_window.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    lib.b2e_attention_causal_d128.restype = i32
    lib.b2e_attention_causal_d128.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.b2e_topk_ip.restype = i32
    lib.b2e_topk_ip.argtypes = [vp, i32, vp, i32, i64, i32, i32, vp, vp, vp]
    lib.b2e_topk_ip_tc.restype = i32
    lib.b2e_topk_ip_tc.argtypes = [vp, i32, vp, i64, i32, i32, C.c_float, vp, vp, vp]
    lib.b2e_max_row_norm.restype = i32
    lib.b2e_max_row_norm.argtypes = [vp, i64, i32, C.POINTER(C.c_float), vp]
    lib.b2e_pack_ubinary.restype = i32
    lib.b2e_pack_ubinary.argtypes = [vp, i64, i32, vp, vp]
    lib.b2e_search_ubinary.restype = i32
    lib.b2e_search_ubinary.argtypes = [vp, i32, vp, i64, i32, i32, i32, vp, vp, vp]
    lib.b2e_layernorm.restype = i32
    lib.b2e_layernorm.argtypes = [vp, vp, vp, vp, i32, i32, C.c_float, i32, vp]


def load(storage: str = 'f16') -> C.CDLL:
    """Load libb2e.so ('f16') or libb2e_bf16.so ('bf16'), once each.  Raises ``NativeError`` when it has not
    been built."""
    if storage in _libs:
        return _libs[storage]
    path = LIB_PATHS[storage]
    if not path.exists():
        raise NativeError(
            f'{path} not found: build it with `python -m distllm_b200.build` '
            '(or __graft_entry__.build()). There is no CPU fallback.',
        )
    try:
        lib = C.CDLL(str(path))
    except OSError as exc:  # pragma: no cover - depends on the box
        raise NativeError(f'cannot load {path}: {exc}') from exc
    _declare(lib)
    want = DTYPE_F16 if storage == 'f16' else DTYPE_BF16
    if lib.b2e_storage_dtype() != want:
        raise NativeError(f'{path} reports storage dtype {lib.b2e_storage_dtype()}, expected {want}')
    _libs[storage] = lib
    return lib


def check(rc: int, lib: C.CDLL | None = None) -> None:
    """Turn a non-zero return code into a NativeError carrying that library's b2e_last_error()."""
    if rc != 0:
        msg = (lib or load()).b2e_last_error()
        raise NativeError(f'libb2e error {rc}: {msg.decode() if msg else "?"}')


def dtype_code(dtype: torch.dtype) -> int:
    try:
        return _DTYPE_CODES[dtype]
    except KeyError:
        raise NativeError(f'unsupported dtype {dtype}') from None


def stream_ptr(device: torch.device | None = None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _cuda_contig(t: torch.Tensor, what: str) -> torch.Tensor:
    if not t.is_cuda:
        raise NativeError(f'{what} must be a CUDA tensor (libb2e has no CPU fallback)')
    if not t.is_contiguous():
        raise NativeError(f'{what} must be contiguous')
    return t


# --------------------------------------------------------------------------- thin op wrappers
def gemm_h16(
    a: torch.Tensor,
    w: torch.Tensor,
    bias: torch.Tensor | None,
    resid: torch.Tensor | None = None,
    epilogue: int = EPI_BIAS,
) -> torch.Tensor:
    """out[M,N] = epi(a[M,K] @ w[N,K].T + bias (+ resid)) on the tcgen05 GEMM; float16 or bfloat16 in/out (the
    matching build of the library is used), fp32 accumulation.

    ``EPI_SWIGLU``: ``w`` holds gate/up rows interleaved in blocks of 64 (weights.interleave_gate_up)
    and the result is ``silu(gate) * up`` of shape [M, N/2]."""
    if a.dtype != w.dtype:
        raise NativeError(f'gemm_h16: operands differ in dtype ({a.dtype} vs {w.dtype})')
    lib = load(storage_of(a.dtype))
    _cuda_contig(a, 'a'), _cuda_contig(w, 'w')
    if bias is not None:
        _cuda_contig(bias, 'bias')
    m, k = a.shape
    n = w.shape[0]
    n_out = n // 2 if epilogue in (EPI_SWIGLU, EPI_GEGLU) else n
    out = torch.empty((m, n_out), dtype=a.dtype, device=a.device)
    with torch.cuda.device(a.device):
        check(lib.b2e_gemm_h16(a.data_ptr(), w.data_ptr(), _ptr(bias), _ptr(resid),
                               out.data_ptr(), m, n, k, epilogue, stream_ptr(a.device)), lib)
    return out


def attention_d64(
    qkv: torch.Tensor,
    attention_mask: torch.Tensor,
    batch: int,
    seq: int,
    heads: int,
) -> torch.Tensor:
    """qkv [B*S, 3*heads*64] fp16 -> context [B*S, heads*64] fp16."""
    lib = load(storage_of(qkv.dtype))
    _cuda_contig(qkv, 'qkv'), _cuda_contig(attention_mask, 'attention_mask')
    ctx = torch.zeros((batch * seq, heads * 64), dtype=qkv.dtype, device=qkv.device)
    with torch.cuda.device(qkv.device):
        check(lib.b2e_attention_d64(qkv.data_ptr(), attention_mask.data_ptr(), ctx.data_ptr(), batch,
                                    seq, heads, None, stream_ptr(qkv.device)), lib)
    return ctx


def attention_d64_window(qkv: torch.Tensor, attention_mask: torch.Tensor, batch: int, seq: int, heads: int,
                         window: int) -> torch.Tensor:
    """Bidirectional sliding-window attention (|i - j| <= window): qkv [B*S, 3*heads*64] fp16 -> [B*S, heads*64]."""
    lib = load(storage_of(qkv.dtype))
    _cuda_contig(qkv, 'qkv'), _cuda_contig(attention_mask, 'attention_mask')
    ctx = torch.zeros((batch * seq, heads * 64), dtype=qkv.dtype, device=qkv.device)
    with torch.cuda.device(qkv.device):
        check(lib.b2e_attention_d64_window(qkv.data_ptr(), attention_mask.data_ptr(), ctx.data_ptr(), batch, seq,
                                           heads, window, stream_ptr(qkv.device)), lib)
    return ctx


def attention_causal_d128(
    qkv: torch.Tensor,
    attention_mask: torch.Tensor,
    batch: int,
    seq: int,
    heads: int,
    kv_heads: int,
    window: int = 0,
) -> torch.Tensor:
    """qkv [B*S, (heads + 2*kv_heads)*128] fp16 (q | k | v, rotary applied) -> [B*S, heads*128] fp16."""
    lib = load(storage_of(qkv.dtype))
    _cuda_contig(qkv, 'qkv'), _cuda_contig(attention_mask, 'attention_mask')
    ctx = torch.zeros((batch * seq, heads * 128), dtype=qkv.dtype, device=qkv.device)
    with torch.cuda.device(qkv.device):
        check(lib.b2e_attention_causal_d128(qkv.data_ptr(), attention_mask.data_ptr(), ctx.data_ptr(),
                                            batch, seq, heads, kv_heads, window, stream_ptr(qkv.device)), lib)
    return ctx


def topk_ip(queries: torch.Tensor, corpus: torch.Tensor, k: int,
            max_norm: float | None = None) -> tuple[torch.Tensor, torch.Tensor]:
    """Exact inner-product top-k: queries [Q,H] f32, corpus [N,H] f32|bf16 (CUDA) -> (scores [Q,k] f32,
    indices [Q,k] i64), sorted by descending score.  ``max_norm`` (an upper bound of the corpus rows' Euclidean
    norms, see :func:`max_row_norm`) selects the tensor-core scan for a float32 corpus; the results are the same."""
    lib = load()
    _cuda_contig(queries, 'queries'), _cuda_contig(corpus, 'corpus')
    if queries.dtype != torch.float32:
        raise NativeError('queries must be float32')
    q, h = queries.shape
    n = corpus.shape[0]
    scores = torch.empty((q, k), dtype=torch.float32, device=queries.device)
    indices = torch.empty((q, k), dtype=torch.int64, device=queries.device)
    with torch.cuda.device(queries.device):
        if max_norm is not None and corpus.dtype == torch.float32:
            check(lib.b2e_topk_ip_tc(queries.data_ptr(), q, corpus.data_ptr(), n, h, k, float(max_norm),
                                     scores.data_ptr(), indices.data_ptr(), stream_ptr(queries.device)))
        else:
            check(lib.b2e_topk_ip(queries.data_ptr(), q, corpus.data_ptr(), dtype_code(corpus.dtype), n, h, k,
                                  scores.data_ptr(), indices.data_ptr(), stream_ptr(queries.device)))
    return scores, indices


def max_row_norm(matrix: torch.Tensor) -> float:
    """Largest Euclidean row norm of a float32 CUDA matrix (index-build step of the tensor-core search)."""
    lib = load()
    _cuda_contig(matrix, 'matrix')
    if matrix.dtype != torch.float32:
        raise NativeError('max_row_norm expects float32')
    out = C.c_float(0.0)
    with torch.cuda.device(matrix.device):
        check(lib.b2e_max_row_norm(matrix.data_ptr(), matrix.shape[0], matrix.shape[1], C.byref(out),
                                   stream_ptr(matrix.device)))
    return float(out.value)


def topk_tc_fell_back() -> bool:
    """Whether this thread's last tensor-core search had to redo the call with the exact scan (debug hook)."""
    lib = load()
    out = C.c_int(0)
    lib.b2e_debug_topk_tc_fell_back.argtypes = [C.POINTER(C.c_int)]
    check(lib.b2e_debug_topk_tc_fell_back(C.byref(out)))
    return bool(out.value)


def debug_pack_layout(attention_mask: torch.Tensor, enable: bool = True, storage: str = 'f16'):
    """Padding-free token layout of a [B, S] int64 mask as the pooled forward pass builds it (debug hook):
    (cu [B+1], len [B], t_real [2], tok_src [B*S]) int32 CUDA tensors.  tok_src starts as -1; only its first
    t_real[0] entries are written."""
    lib = load(storage)
    _cuda_contig(attention_mask, 'attention_mask')
    if attention_mask.dtype != torch.int64:
        raise NativeError('attention_mask must be int64')
    b, s = attention_mask.shape
    dev = attention_mask.device
    cu = torch.full((b + 1,), -1, dtype=torch.int32, device=dev)
    ln = torch.full((b,), -1, dtype=torch.int32, device=dev)
    t_real = torch.full((2,), -1, dtype=torch.int32, device=dev)
    tok_src = torch.full((b * s,), -1, dtype=torch.int32, device=dev)
    lib.b2e_debug_pack_layout.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 5
    with torch.cuda.device(dev):
        check(lib.b2e_debug_pack_layout(attention_mask.data_ptr(), b, s, int(enable), cu.data_ptr(), ln.data_ptr(),
                                        t_real.data_ptr(), tok_src.data_ptr(), stream_ptr(dev)), lib)
    return cu, ln, t_real, tok_src


def debug_gemm_rows(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor | None, resid: torch.Tensor | None,
                    epilogue: int, m_dev: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """:func:`gemm_h16` into ``out`` with the row count read from the device int32 ``m_dev`` (debug hook): row
    tiles at or beyond it are left alone."""
    lib = load(storage_of(a.dtype))
    for t, what in ((a, 'a'), (w, 'w'), (out, 'out'), (m_dev, 'm_dev')):
        _cuda_contig(t, what)
    if m_dev.dtype != torch.int32:
        raise NativeError('m_dev must be int32')
    m, k = a.shape
    n = w.shape[0]
    lib.b2e_debug_gemm_rows.argtypes = [C.c_void_p] * 5 + [C.c_int] * 4 + [C.c_void_p] * 2
    with torch.cuda.device(a.device):
        check(lib.b2e_debug_gemm_rows(a.data_ptr(), w.data_ptr(), _ptr(bias), _ptr(resid), out.data_ptr(), m, n, k,
                                      epilogue, m_dev.data_ptr(), stream_ptr(a.device)), lib)
    return out


def debug_attention_packed(qkv: torch.Tensor, attention_mask: torch.Tensor, cu: torch.Tensor, seq_len: torch.Tensor,
                           ctx: torch.Tensor, heads: int, kv_heads: int, head_dim: int, window: int = 0) -> torch.Tensor:
    """Attention on the packed token layout (debug hook): sequence b in rows cu[b] .. cu[b]+len[b]-1 of ``qkv`` and
    ``ctx`` (both B*S rows).  head_dim 64: the bidirectional / sliding-window kernel; 128: causal grouped-query."""
    lib = load(storage_of(qkv.dtype))
    for t, what in ((qkv, 'qkv'), (attention_mask, 'attention_mask'), (cu, 'cu'), (seq_len, 'len'), (ctx, 'ctx')):
        _cuda_contig(t, what)
    b, s = attention_mask.shape
    lib.b2e_debug_attention_packed.argtypes = [C.c_void_p] * 5 + [C.c_int] * 6 + [C.c_void_p]
    with torch.cuda.device(qkv.device):
        check(lib.b2e_debug_attention_packed(qkv.data_ptr(), attention_mask.data_ptr(), cu.data_ptr(),
                                             seq_len.data_ptr(), ctx.data_ptr(), b, s, heads, kv_heads, head_dim,
                                             window, stream_ptr(qkv.device)), lib)
    return ctx


def pack_ubinary(embeddings: torch.Tensor) -> torch.Tensor:
    """fp32 [N,H] (CUDA) -> uint8 [N,H/8]: bit = value > 0, first dimension in the most significant bit."""
    lib = load()
    _cuda_contig(embeddings, 'embeddings')
    if embeddings.dtype != torch.float32:
        raise NativeError('pack_ubinary expects float32')
    n, h = embeddings.shape
    out = torch.empty((n, h // 8), dtype=torch.uint8, device=embeddings.device)
    with torch.cuda.device(embeddings.device):
        check(lib.b2e_pack_ubinary(embeddings.data_ptr(), n, h, out.data_ptr(), stream_ptr(embeddings.device)))
    return out


def search_ubinary(queries: torch.Tensor, corpus_bits: torch.Tensor, k: int,
                   rescore_multiplier: int = 2) -> tuple[torch.Tensor, torch.Tensor]:
    """Hamming top-(k * rescore_multiplier) over packed bits + float rescoring: (scores [Q,k] f32,
    indices [Q,k] i64), descending score."""
    lib = load()
    _cuda_contig(queries, 'queries'), _cuda_contig(corpus_bits, 'corpus_bits')
    if queries.dtype != torch.float32 or corpus_bits.dtype != torch.uint8:
        raise NativeError('search_ubinary expects float32 queries and a uint8 packed corpus')
    q, h = queries.shape
    n = corpus_bits.shape[0]
    if corpus_bits.shape[1] * 8 != h:
        raise NativeError(f'corpus has {corpus_bits.shape[1] * 8} bits per row, queries have {h} dimensions')
    scores = torch.empty((q, k), dtype=torch.float32, device=queries.device)
    indices = torch.empty((q, k), dtype=torch.int64, device=queries.device)
    with torch.cuda.device(queries.device):
        check(lib.b2e_search_ubinary(queries.data_ptr(), q, corpus_bits.data_ptr(), n, h, k, rescore_multiplier,
                                     scores.data_ptr(), indices.data_ptr(), stream_ptr(queries.device)))
    return scores, indices


def layernorm(
    x: torch.Tensor,
    gamma: torch.Tensor,
    beta: torch.Tensor,
    eps: float,
    out_dtype: torch.dtype | None = None,
) -> torch.Tensor:
    """LayerNorm of a 16-bit matrix; ``out_dtype``: float32 or (default) the input's own 16-bit type."""
    lib = load(storage_of(x.dtype))
    out_dtype = out_dtype or x.dtype
    _cuda_contig(x, 'x')
    rows, h = x.shape
    out = torch.empty((rows, h), dtype=out_dtype, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.b2e_layernorm(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows,
                                h, eps, dtype_code(out_dtype), stream_ptr(x.device)), lib)
    return out


def pool_mean(
    hidden: torch.Tensor,
    attention_mask: torch.Tensor,
    pool_kind: int = POOL_MEAN_REF,
    mutate_mask: bool = True,
) -> torch.Tensor:
    """Masked mean over the sequence axis; fp32 [B,H].  Rewrites the mask like the reference."""
    lib = load()
    _cuda_contig(hidden, 'hidden'), _cuda_contig(attention_mask, 'attention_mask')
    if attention_mask.dtype != torch.int64:
        raise NativeError('attention_mask must be int64')
    b, s, h = hidden.shape
    out = torch.empty((b, h), dtype=torch.float32, device=hidden.device)
    with torch.cuda.device(hidden.device):
        check(lib.b2e_pool_mean(hidden.data_ptr(), dtype_code(hidden.dtype), attention_mask.data_ptr(),
                                b, s, h, pool_kind, int(mutate_mask), out.data_ptr(),
                                stream_ptr(hidden.device)))
    return out


def pool_last_token(hidden: torch.Tensor, attention_mask: torch.Tensor) -> torch.Tensor:
    lib = load()
    _cuda_contig(hidden, 'hidden'), _cuda_contig(attention_mask, 'attention_mask')
    if attention_mask.dtype != torch.int64:
        raise NativeError('attention_mask must be int64')
    b, s, h = hidden.shape
    out = torch.empty((b, h), dtype=torch.float32, device=hidden.device)
    with torch.cuda.device(hidden.device):
        check(lib.b2e_pool_last_token(hidden.data_ptr(), dtype_code(hidden.dtype),
                                      attention_mask.data_ptr(), b, s, h, out.data_ptr(),
                                      stream_ptr(hidden.device)))
    return out


def l2_normalize_(x: torch.Tensor) -> torch.Tensor:
    lib = load()
    _cuda_contig(x, 'x')
    if x.dtype != torch.float32:
        raise NativeError('l2_normalize_ expects fp32')
    n, h = x.shape
    with torch.cuda.device(x.device):
        check(lib.b2e_l2_normalize(x.data_ptr(), n, h, stream_ptr(x.device)))
    return x


def adjacent_cosine_dist(emb: torch.Tensor, doc_id: torch.Tensor | None = None) -> torch.Tensor:
    """fp32 [N-1]: 1 - cos(emb[i], emb[i+1]); NaN where doc_id changes."""
    lib = load()
    _cuda_contig(emb, 'emb')
    n, h = emb.shape
    out = torch.empty((max(n - 1, 0),), dtype=torch.float32, device=emb.device)
    if doc_id is not None:
        _cuda_contig(doc_id, 'doc_id')
        if doc_id.dtype != torch.int32:
            raise NativeError('doc_id must be int32')
    with torch.cuda.device(emb.device):
        check(lib.b2e_adjacent_cosine_dist(emb.data_ptr(), dtype_code(emb.dtype), n, h,
                                           _ptr(doc_id), out.data_ptr(), stream_ptr(emb.device)))
    return out
