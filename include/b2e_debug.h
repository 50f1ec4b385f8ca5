/* b2e_debug.h -- profiling / experiment hooks of libb2e.so.
 *
 * NOT part of the reference-facing ABI (include/b2e.h): nothing in distllm would bind these.  They
 * exist for the timeline tools under tools/ (att3_timeline.py, gemm_timeline.py, pair_experiments.py)
 * and are declared here so that every symbol the shared library exports is declared in a header.
 * The set_* hooks write a __device__ global of the kernels' translation unit; the test hooks at the end launch
 * kernels on caller buffers (tests/).  All return 0 on success.
 */
#ifndef B2E_DEBUG_H_
#define B2E_DEBUG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

struct B2EEncoder;
/* run only the first n layers of an encoder handle from now on (0 = full depth again): the per-layer
 * drift report (tools/drift_report.py) compares every depth with the CPU oracle */
int b2e_debug_set_layers(struct B2EEncoder* enc, int n_layers);

/* device buffer of 4 x 512 int64: CTA 0 of the streaming attention kernels records (clock64, event
 * code) pairs per role (softmax slot A/B, MMA issuer, loader); NULL switches it off */
int b2e_debug_set_att3_clock(void* device_buffer);
/* scheduling experiments of the attention kernels (attention3.cuh g_att3_flags): bits 0-1 ordering of the two
 * softmax warpgroups (0 free-running, 1 strict ping-pong, 2 de-phased once per item = default), bit 2 the loader
 * and MMA-issuer threads wait parked in hardware (mbarrier.try_wait with a suspend-time hint) instead of polling */
int b2e_debug_set_att3_flags(int flags);
/* 0: keep the padded [B, S] token layout on every path; 1 (default, also B2E_PACKED=1): pooled forward passes run
 * on the attended tokens only (csrc/pack.cuh).  Drops the handle's cached CUDA graphs' validity: call it before
 * b2e_embed_host, not between its batches. */
int b2e_debug_set_packing(int on);
/* *out = 1 when this thread's last b2e_topk_ip_tc call had to fall back to the exact scan (synchronises the device) */
int b2e_debug_topk_tc_fell_back(int* out);
/* which instantiated softmax variant of attention3_d64_kernel<V> the next launches use (also B2E_ATT3) */
int b2e_debug_set_att3_variant(int variant);
/* CTA-pair GEMM: bit 0 = skip the epilogue's math and stores (experiment) */
int b2e_debug_set_pair_flags(int flags);
/* device buffer of 4 x 256 int64 filled with clock64() stamps by CTAs 0/1 of the CTA-pair GEMM */
int b2e_debug_set_clock_buffer(void* device_buffer);

/* Test hooks of the padding-free ("packed") token layout (csrc/pack.cuh), used by tests/.  Pointers are device
 * pointers; every call is asynchronous on `stream`.
 *
 * The layout the pooled forward pass builds from an int64 [B, S] mask: cu [B + 1], len [B], t_real [2] (rows in
 * use, packed flag) and tok_src [B * S] (only its first t_real[0] entries are written).  enable = 0 forces the
 * identity layout. */
int b2e_debug_pack_layout(const int64_t* mask, int B, int S, int enable, int* cu, int* len, int* t_real,
                          int* tok_src, void* stream);
/* b2e_gemm_h16 with the row count m_dev (device int, <= M) read on the device: row tiles at or beyond it are
 * skipped; M sizes the grid and the tensor maps */
int b2e_debug_gemm_rows(const void* A, const void* W, const float* bias, const void* resid, void* out, int M,
                        int N, int K, int epi, const int* m_dev, void* stream);
/* attention on the packed layout: qkv and ctx hold B*S rows, sequence b in rows cu[b] .. cu[b] + len[b] - 1.
 * head_dim 64: bidirectional (window 0) or sliding-window attention, kv_heads == heads, the variant of
 * b2e_debug_set_att3_variant; head_dim 128: causal grouped-query attention (window 0 = none). */
int b2e_debug_attention_packed(const void* qkv, const int64_t* mask, const int* cu, const int* len, void* ctx,
                               int B, int S, int heads, int kv_heads, int head_dim, int window, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2E_DEBUG_H_ */
