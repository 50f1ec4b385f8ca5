"""Benchmark of the embedding hot path: embedded chunks/s at 512 tokens (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], "C2"): S-PubMedBert-MS-MARCO shape (BERT-base: L=12, H=768,
12 heads, I=3072, vocab 30522), mean pooler, batch_size=512, 512-token chunks, synthetic
pre-tokenised ids, seeded random-init weights (no checkpoint can be downloaded here).

A step = one pass of the hot path over one batch of 512 chunks per rank: forward pass, fused
reference-semantics mean pool, and the semantic splitter's adjacent-cosine kernel over the step's
pooled rows.  Ranks shard the chunk stream (weak scaling: 512 chunks per rank per step) and meet in
one NCCL all-gather of the pooled matrix at the end of the timed region.

Printed JSON (one line, rank 0):
  value      chunks/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        chunks/s through the C-ABI host-buffer call (b2e_embed_host): pinned host ids/mask in,
             H2D + compute + D2H of the pooled rows inside the timed region; at N > 1 the all-gather of
             the ranks' result matrices is inside it too
  roofline   tensor-core bound: the dominant kernel (FFN-up GEMM) timed alone with CUDA events against
             the measured burst bf16 peak, its DRAM traffic per launch from the committed ncu capture
             (profiles/ncu_traffic.json), and under "whole_step" the step-level achieved TFLOP/s
             (algorithmic matmul FLOPs, SURVEY 8d) against the measured sustained bf16 peak
  cpu_baseline  the UNMODIFIED reference (oracle/_ref: `distllm.distributed_embedding.embedding_worker`,
             its own `[timer] [computed-embeddings ...]` reading) on this box's host cores on a bounded
             sample, in a CPU-only subprocess (rank 0, N=1 only); plus the cosine between its embeddings
             and this repository's for the same checkpoint and file.  Falls back to the oracle port
             (kind "port") when oracle/_ref is absent.
  extra      the other BASELINE configs and the plugin-level numbers, each with its own roofline fraction:
             ragged (lengths ~U{64..512}), c5_esm2_650m (S=1026), c3_mistral7b (B=16, S=4096),
             c4_gather (N > 1: >= 2 M rows per rank through the all-gather), e2e_worker (tokeniser ->
             embedding_worker -> writer), c1 (1 000 x 128-token chunks, batch 8, through the worker)
--impl reference times the unmodified reference as its own arm (rank 0 only; CUDA hidden from it).
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

# the reference arm is the reference's CPU path: it moves its model to CUDA whenever a device is visible
# (distllm/embed/encoders/auto.py:86-90), so the devices are hidden BEFORE torch initialises
if '--impl=reference' in sys.argv or (
        '--impl' in sys.argv and sys.argv[sys.argv.index('--impl') + 1:][:1] == ['reference']):
    os.environ['CUDA_VISIBLE_DEVICES'] = ''

import torch  # noqa: E402

from tools import workloads  # noqa: E402

SEQ = 512
BATCH = 512
BERT_BASE = workloads.BERT_BASE
WORKLOAD = ('C2: S-PubMedBert-MS-MARCO shape (BERT-base L12 H768 I3072), mean pooler (reference '
            'semantics), batch_size=512, 512-token chunks, pre-tokenised synthetic ids, random-init weights')
METRIC = 'embedded chunks/sec @512-tok'
FALLBACK_PEAKS = {'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'hbm_gbs': 6650.0}
ESM2_650M = dict(vocab_size=33, hidden_size=1280, num_hidden_layers=33, num_attention_heads=20,
                 intermediate_size=5120, max_position_embeddings=1026, position_embedding_type='rotary',
                 token_dropout=True, mask_token_id=32, pad_token_id=1, layer_norm_eps=1e-5,
                 emb_layer_norm_before=False, initializer_range=0.02)
MISTRAL_7B = dict(vocab_size=32000, hidden_size=4096, num_hidden_layers=32, num_attention_heads=32,
                  num_key_value_heads=8, head_dim=128, intermediate_size=14336,
                  max_position_embeddings=32768, rms_norm_eps=1e-5, sliding_window=4096,
                  initializer_range=0.02)


def flops_per_chunk(cfg: dict, s: int) -> float:
    """Algorithmic matmul FLOPs (SURVEY.md 8d): L * (8 S H^2 + 4 S H I + 4 S^2 H)."""
    h, i, layers = cfg['hidden_size'], cfg['intermediate_size'], cfg['num_hidden_layers']
    return layers * (8.0 * s * h * h + 4.0 * s * h * i + 4.0 * s * s * h)


def mistral_flops_per_seq(cfg: dict, s: int, causal_skipped: bool = True) -> float:
    """SURVEY 8d: 4SH^2 (q,o) + 4 S H (kv_heads d) (k,v) + 6 S H I + attention (dense 4 S^2 H, or the
    causal-skipped 2 S (S+128) H that the kernel's chunk skipping actually executes)."""
    h, i, layers = cfg['hidden_size'], cfg['intermediate_size'], cfg['num_hidden_layers']
    qc = (cfg['num_attention_heads'] + 2 * cfg['num_key_value_heads']) * cfg['head_dim']
    att = 2.0 * s * (s + 128) * h if causal_skipped else 4.0 * s * s * h
    return layers * (2.0 * s * h * qc + 2.0 * s * h * h + 6.0 * s * h * i + att)


def launches_per_step(cfg: dict) -> int:
    """Kernels of ours per step: the 3 kernels of the padding-free layout (lengths, scan, row map), embed+LN,
    attention mask prep, per layer 4 GEMMs + attention + 2 LayerNorms (the last LayerNorm is the fused LN+pool),
    3 pool-weight kernels, pool finalize, adjacent-cosine (matches profiles/r02_ncu_launches_final.md: 1413
    launches in 15 passes)."""
    return 3 + 1 + 1 + cfg['num_hidden_layers'] * 7 + 3 + 1 + 1


def load_peaks() -> tuple[dict, str]:
    path = REPO / 'MEASURED_PEAKS.json'
    if path.exists():
        return json.loads(path.read_text()), 'measured'
    return dict(FALLBACK_PEAKS), 'fallback'


def synthetic_batch(n: int, s: int, vocab: int, seed: int, ragged: tuple[int, int] | None = None):
    """ids ~ U{7..V-1} with [CLS]=101 first / [SEP]=102 last, zero token types; all-ones mask, or (ragged)
    right-padded rows with lengths ~ U{lo..hi} and the first row at full length."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(7, vocab, (n, s), generator=g, dtype=torch.int64)
    ids[:, 0] = 101
    if ragged is None:
        ids[:, -1] = 102
        return ids, torch.ones(n, s, dtype=torch.int64), torch.zeros(n, s, dtype=torch.int64)
    lens = torch.randint(ragged[0], ragged[1] + 1, (n,), generator=g)
    lens[0] = s
    mask = (torch.arange(s)[None] < lens[:, None]).long()
    ids[torch.arange(n), lens - 1] = 102
    ids = ids * mask
    return ids, mask, torch.zeros(n, s, dtype=torch.int64)


class ClockSampler:
    """nvidia-smi clock/throttle sampling during the timed region (recipe in B200_PROFILING.md)."""

    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index: int) -> None:
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self) -> None:
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.gpu_index}', f'--query-gpu={self.QUERY}',
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for line in Path(self.path).read_text().splitlines():
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        busy = sorted(sm)[len(sm) // 4:] if len(sm) >= 4 else sm  # drop idle samples at the edges
        return {'sm_mhz': statistics.median(busy), 'sm_max_mhz': max(smax), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ===================================================================================== reference arm
def worker_kwargs(ckpt: Path, batch: int, dataset: str = 'jsonl', embedder: str = 'full_sequence',
                  workers: int = 4, **extra) -> dict:
    """kwargs of `embedding_worker` (same keys on both arms): the CLI's own mapping
    (distllm/cli.py:124-173) with fp32, quantization off, eval mode."""
    dataset_kwargs = {'name': dataset, 'batch_size': batch, 'num_data_workers': workers}
    if dataset == 'jsonl_chunk':
        dataset_kwargs['buffer_size'] = extra.get('buffer_size', 4)
    embedder_kwargs = {'name': embedder}
    if embedder == 'semantic_chunk':
        embedder_kwargs['chunk_batch_size'] = extra.get('chunk_batch_size', batch)
    return dict(
        dataset_kwargs=dataset_kwargs,
        encoder_kwargs={'name': 'auto', 'pretrained_model_name_or_path': str(ckpt), 'half_precision': False,
                        'eval_mode': True, 'compile_model': False, 'quantization': False},
        pooler_kwargs={'name': 'mean'},
        embedder_kwargs=embedder_kwargs,
        writer_kwargs={'name': 'numpy'},
    )


def reference_available() -> bool:
    from oracle import ref_shims

    return ref_shims.reference_root() is not None


def _pick_reference_threads(run_once) -> int:
    """The thread count at which the CPU arm is fastest (all schedulable CPUs, then halves): torch CPU
    GEMMs are not always best with every SMT sibling busy.  A process-wide torch setting, not a change to
    the reference."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    best, best_t = avail, float('inf')
    for n in sorted({max(1, avail >> k) for k in range(0, 3)}, reverse=True):
        torch.set_num_threads(n)
        run_once()   # warm this thread count
        sec = run_once()
        if sec < best_t:
            best, best_t = n, sec
    torch.set_num_threads(best)
    return best


def run_reference(args) -> None:
    """The unmodified reference on the host CPUs: each step is one `embedding_worker` call
    (distllm/distributed_embedding.py:23-80) over a file of `--sample-chunks` chunks of 512 tokens, batch 8
    (the reference's default), `jsonl` dataset, `full_sequence` embedder, `mean` pooler, `numpy` writer; the
    step time is the reference's own `[timer] [computed-embeddings <file>]` line."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if not reference_available():
        run_reference_port(args)
        return
    from oracle import ref_shims

    per_step = args.sample_chunks
    with tempfile.TemporaryDirectory(prefix='b2e_ref_') as tmp:
        tmp = Path(tmp)
        ckpt = Path(args.checkpoint) if args.checkpoint else workloads.write_bert_checkpoint(tmp / 'ckpt')
        step_file = Path(args.sample_file) if args.sample_file else workloads.write_token_rows(
            tmp / 'c2_sample.jsonl', per_step, SEQ, BERT_BASE['vocab_size'], seed=123)
        tiny = workloads.write_token_rows(tmp / 'tiny.jsonl', 2, SEQ, BERT_BASE['vocab_size'], seed=5)
        kw = worker_kwargs(ckpt, batch=8, workers=args.data_workers)
        n = [0]
        last_out = [tmp]

        def run(path: Path) -> dict:
            n[0] += 1
            last_out[0] = tmp / f'out{n[0]}'
            return ref_shims.run_embedding_worker(path, last_out[0], **kw)

        run(tiny)   # loads the encoder into the reference's registry (warm start, registry.py:90-132)
        threads = _pick_reference_threads(lambda: run(tiny)['computed-embeddings'])
        for _ in range(args.warmup):
            run(step_file)
        times = [run(step_file)['computed-embeddings'] for _ in range(args.steps)]
        step_out = last_out[0]
        total = sum(times)
        value = per_step * args.steps / total
        sample = (f'{args.steps} x embedding_worker over {per_step} chunks of {SEQ} tokens (batch 8, jsonl + '
                  f'full_sequence + mean + numpy writer, {args.data_workers} DataLoader workers), fp32 torch CPU; '
                  f"the reference's own [timer] [computed-embeddings] seconds")
        extra = {}
        if args.with_c1:
            # BASELINE config C1 exactly as written: 1 000 synthetic 128-token chunks, batch 8, CPU
            c1 = workloads.write_token_rows(tmp / 'c1.jsonl', 1000, 128, BERT_BASE['vocab_size'], seed=1)
            sec = run(c1)['computed-embeddings']
            extra['c1'] = {'workload': 'C1: 1 000 x 128-token chunks, mean pooler, batch_size=8, CPU',
                           'value': 1000 / sec, 'unit': 'chunks/s', 'seconds': sec, 'cores': threads}
        if args.embeddings_out:
            import shutil

            shutil.copy(next(step_out.glob('*/embeddings.npy')), args.embeddings_out)
        line = {
            'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'chunks/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': 1e3 * total / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'global_batch': 8, 'seq_len': SEQ, 'parallelism': 'cpu',
                       'sample_chunks_per_step': per_step},
            'cpu_baseline': {'value': value, 'unit': 'chunks/s', 'cores': threads, 'kind': 'reference',
                             'sample': sample, 'reference_root': str(ref_shims.reference_root())},
            'e2e': {'value': value, 'unit': 'chunks/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0, 'extra': extra,
        }
        emit(line, args.json_out)


_CPU_WEIGHTS: dict = {}


def cpu_oracle_run(n_chunks: int, batch: int, seed: int = 0):
    """FALLBACK when oracle/_ref is absent: time the CPU port of the reference path (oracle forward +
    reference mean pool) on ``n_chunks`` synthetic 512-token chunks.  Returns (seconds, chunks)."""
    from transformers import BertConfig

    from distllm_b200.embed.encoders.weights import random_bert_state_dict
    from oracle import bert as obert
    from oracle import pooling as opool

    cfg = BertConfig(**BERT_BASE)
    if seed not in _CPU_WEIGHTS:
        _CPU_WEIGHTS[seed] = random_bert_state_dict(cfg, seed=seed, device='cpu')
    sd = _CPU_WEIGHTS[seed]
    ids, mask, types = synthetic_batch(n_chunks, SEQ, BERT_BASE['vocab_size'], seed=123)
    obert.bert_forward(sd, cfg, ids[:1], mask[:1], types[:1])
    t0 = time.perf_counter()
    for lo in range(0, n_chunks, batch):
        hidden = obert.bert_forward(sd, cfg, ids[lo:lo + batch], mask[lo:lo + batch], types[lo:lo + batch])
        opool.average_pool(hidden, mask[lo:lo + batch].clone())
    return time.perf_counter() - t0, n_chunks


def run_reference_port(args) -> None:
    per_step = args.sample_chunks
    threads = _pick_reference_threads(lambda: cpu_oracle_run(2, 2)[0])
    if args.warmup > 0:
        cpu_oracle_run(per_step, 8)
    total = sum(cpu_oracle_run(per_step, 8)[0] for _ in range(args.steps))
    value = per_step * args.steps / total
    sample = f'{args.steps} steps x {per_step} chunks of {SEQ} tokens (batch 8), fp32 torch CPU port (oracle/)'
    emit({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'chunks/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'global_batch': 8, 'seq_len': SEQ, 'parallelism': 'cpu',
                   'sample_chunks_per_step': per_step},
        'cpu_baseline': {'value': value, 'unit': 'chunks/s', 'cores': threads, 'kind': 'port', 'sample': sample,
                         'note': 'oracle/_ref absent: the oracle port ran instead of the reference'},
        'e2e': {'value': value, 'unit': 'chunks/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }, args.json_out)


# ======================================================================================== native arm
def time_dominant_kernel(device: torch.device, peaks: dict, dtype: torch.dtype = torch.bfloat16) -> dict:
    """FFN-up GEMM (M=B*S, N=3072, K=768, bias+GELU epilogue) timed alone with CUDA events, in the build of the
    library whose 16-bit storage type is ``dtype`` (the BERT family runs the bfloat16 build)."""
    from distllm_b200 import _native as nv

    m, n, k = BATCH * SEQ, BERT_BASE['intermediate_size'], BERT_BASE['hidden_size']
    a = torch.randn(m, k, device=device).to(dtype)
    w = (torch.randn(n, k, device=device) * 0.02).to(dtype)
    bias = torch.zeros(n, device=device)
    for _ in range(3):
        nv.gemm_h16(a, w, bias, None, nv.EPI_BIAS_GELU)
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(device)
    e0.record()
    for _ in range(reps):
        nv.gemm_h16(a, w, bias, None, nv.EPI_BIAS_GELU)
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / reps
    tf = 2.0 * m * n * k / (ms * 1e-3) / 1e12
    return {'name': DOMINANT_KERNEL, 'flops_per_launch': 2.0 * m * n * k,
            'ms_per_launch': ms, 'achieved': tf, 'peak': peaks['bf16_tflops'], 'frac': tf / peaks['bf16_tflops'],
            'unit': 'TFLOP/s', 'peak_kind': 'burst (kernel timed alone)'}


def storage_ab(device: torch.device) -> dict:
    """The same FFN-up GEMM in the two builds of the library, long enough (about 1.5 s each) to reach the
    power-capped clock: what the 16-bit storage type costs in sustained tensor throughput."""
    from distllm_b200 import _native as nv

    m, n, k = BATCH * SEQ, BERT_BASE['intermediate_size'], BERT_BASE['hidden_size']
    out = {}
    for name, dtype in (('bf16', torch.bfloat16), ('f16', torch.float16), ('bf16_again', torch.bfloat16)):
        a = torch.randn(m, k, device=device).to(dtype)
        w = (torch.randn(n, k, device=device) * 0.02).to(dtype)
        bias = torch.zeros(n, device=device)
        for _ in range(300):   # ~0.3 s to settle the clock
            nv.gemm_h16(a, w, bias, None, nv.EPI_BIAS_GELU)
        reps = 1200
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(device)
        e0.record()
        for _ in range(reps):
            nv.gemm_h16(a, w, bias, None, nv.EPI_BIAS_GELU)
        e1.record()
        torch.cuda.synchronize(device)
        ms = e0.elapsed_time(e1) / reps
        out[name] = {'ms_per_launch': ms, 'tflops': 2.0 * m * n * k / (ms * 1e-3) / 1e12}
    out['what'] = 'FFN-up GEMM (M=262144 N=3072 K=768, bias + GELU), 1200 back-to-back launches per storage type'
    return out


DOMINANT_KERNEL = 'gemm2_h16_pair<5,GELU> (FFN up, M=262144 N=3072 K=768; CTA-pair tcgen05 kernel, bfloat16 build)'


def ncu_traffic_bytes() -> float | None:
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the
    committed `ncu --set full` summary (profiles/ncu_traffic.json, written by tools/ncu_traffic.py)."""
    path = REPO / 'profiles' / 'ncu_traffic.json'
    if not path.exists():
        return None
    return json.loads(path.read_text()).get('ffn_up_gemm_b512', {}).get('dram_bytes_per_launch')


def timed_steps(fn, steps: int, warm: int, device) -> float:
    """ms per call of ``fn`` (CUDA events on the current stream, after ``warm`` untimed calls)."""
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(device)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(device)
    return e0.elapsed_time(e1) / steps


def extra_esm2(device, peaks: dict, reduce_max) -> dict:
    """BASELINE C5: ESM2-650M shape, 1024 residues -> S=1026, mean pooler, batch 64 per rank."""
    from transformers import EsmConfig

    from distllm_b200 import _native as nv
    from distllm_b200.embed.encoders.native import NativeEsm2Encoder
    from distllm_b200.embed.encoders.weights import random_esm_state_dict

    cfg = EsmConfig(**ESM2_650M)
    b, s = 64, 1026
    enc = NativeEsm2Encoder(cfg, random_esm_state_dict(cfg, seed=0, device=device), device=device)
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(4, 24, (b, s), generator=g)
    ids[:, 0], ids[:, -1] = 0, 2
    ids = ids.to(device)
    mask = torch.ones(b, s, dtype=torch.int64, device=device)
    out = torch.empty(b, cfg.hidden_size, device=device)
    ms = reduce_max(timed_steps(lambda: enc.encode_pooled(ids, mask, None, nv.POOL_MEAN_REF, False, out=out),
                                5, 3, device))
    enc.close()
    del enc
    torch.cuda.empty_cache()
    seqs = b / (ms * 1e-3)
    tf = seqs * flops_per_chunk(ESM2_650M, s) / 1e12
    return {'workload': 'C5: ESM2-650M shape (L33 H1280 I5120), 1024 residues -> S=1026, mean pooler, '
                        'batch 64 per GPU, synthetic residues, random-init weights; bfloat16-storage build',
            'value_per_gpu': seqs, 'unit': 'sequences/s', 'ms_per_step': ms, 'steps': 5,
            'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peaks['bf16_tflops_sustained'],
                         'unit': 'TFLOP/s', 'frac': tf / peaks['bf16_tflops_sustained'],
                         'flops_per_sequence': flops_per_chunk(ESM2_650M, s)}}


def extra_retrieval(device, peaks: dict) -> dict:
    """SURVEY 8(f) rank 2, the consumer of the gathered matrix: exact inner-product search of 16 queries, k = 100,
    over a device-resident 1 M x 768 float32 matrix (3.1 GB: far beyond L2) -- CUDA-core scan vs the tensor-core
    scan with exact fp32 decision; both must name the same rows."""
    from distllm_b200 import _native as nv

    n, h, q, k = 1_000_000, 768, 16, 100
    g = torch.Generator(device=device).manual_seed(3)
    corpus = torch.randn(n, h, device=device, generator=g)
    corpus = (corpus / corpus.norm(dim=1, keepdim=True)).contiguous()
    queries = torch.randn(q, h, device=device, generator=g)
    queries = queries / queries.norm(dim=1, keepdim=True)
    max_norm = nv.max_row_norm(corpus) * 1.0001
    out = {'workload': f'{q} queries, k={k}, corpus {n} x {h} float32 L2-normalised rows on the device',
           'algorithmic_bytes': n * h * 4, 'hbm_peak_gbs': peaks['hbm_gbs']}
    ref = None
    for name, kw in (('cuda_core_scan', {}), ('tensor_core_scan', {'max_norm': max_norm})):
        res = nv.topk_ip(queries, corpus, k, **kw)
        ms = timed_steps(lambda: nv.topk_ip(queries, corpus, k, **kw), 5, 2, device)
        gbs = n * h * 4 / ms / 1e6
        out[name] = {'ms': ms, 'queries_per_s': q / ms * 1e3, 'gb_per_s': gbs, 'frac_of_hbm': gbs / peaks['hbm_gbs']}
        if ref is None:
            ref = res
        else:
            out[name]['same_rows_as_cuda_core_scan'] = bool(torch.equal(res[1], ref[1]))
            out[name]['fell_back_to_exact_scan'] = nv.topk_tc_fell_back()
    del corpus
    torch.cuda.empty_cache()
    return out


def extra_mistral(device, peaks: dict, reduce_max) -> dict:
    """BASELINE C3: SFR-Embedding-Mistral shape (Mistral-7B), last_token pooler, batch 16, S=4096."""
    from transformers import MistralConfig

    from distllm_b200 import _native as nv
    from distllm_b200.embed.encoders.native import NativeMistralEncoder
    from distllm_b200.embed.encoders.weights import random_mistral_state_dict

    cfg = MistralConfig(**MISTRAL_7B)
    b, s = 16, 4096
    sd = random_mistral_state_dict(cfg, seed=0, device=device, dtype=torch.float16)
    enc = NativeMistralEncoder(cfg, sd, device=device)
    del sd
    torch.cuda.empty_cache()
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(3, 32000, (b, s), generator=g).to(device)
    mask = torch.ones(b, s, dtype=torch.int64, device=device)
    out = torch.empty(b, cfg.hidden_size, device=device)
    ms = reduce_max(timed_steps(lambda: enc.encode_pooled(ids, mask, None, nv.POOL_LAST_TOKEN, True, out=out),
                                3, 2, device))
    # the same batch shape with right-padded lengths ~ U{512..4096} (first row full): the padding-free layout makes
    # the step cost what its attended tokens cost
    lens = torch.randint(s // 8, s + 1, (b,), generator=g)
    lens[0] = s
    r_mask = (torch.arange(s)[None] < lens[:, None]).long().to(device)
    r_ms = reduce_max(timed_steps(lambda: enc.encode_pooled(ids, r_mask, None, nv.POOL_LAST_TOKEN, True, out=out),
                                  2, 1, device))
    ragged = {'workload': 'same model and batch shape, lengths ~ U{512..4096} right-padded', 'ms_per_step': r_ms,
              'sequences_per_s_per_gpu': b / (r_ms * 1e-3), 'attended_tokens': int(r_mask.sum().item()),
              'padded_tokens': b * s}
    enc.close()
    del enc
    torch.cuda.empty_cache()
    seqs = b / (ms * 1e-3)
    tf = seqs * mistral_flops_per_seq(MISTRAL_7B, s) / 1e12
    return {'ragged': ragged,
            'workload': 'C3: SFR-Embedding-Mistral shape (Mistral-7B: L32 H4096 32q/8kv x128 I14336), '
                        'last_token pooler, batch_size=16, S=4096, synthetic ids, random-init weights; half-storage build (f16)',
            'value_per_gpu': seqs, 'unit': 'sequences/s', 'ms_per_step': ms, 'steps': 3,
            'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peaks['bf16_tflops_sustained'],
                         'unit': 'TFLOP/s', 'frac': tf / peaks['bf16_tflops_sustained'],
                         'flops_per_sequence': mistral_flops_per_seq(MISTRAL_7B, s),
                         'flops_counted': 'causal-skipped attention (2 S (S+128) H per layer), SURVEY 8d',
                         'dense_counted_tflops': seqs * mistral_flops_per_seq(MISTRAL_7B, s, False) / 1e12}}


def extra_worker(device, rank: int, world: int, reduce_max, do_c1: bool) -> dict:
    """Plugin level: files on disk -> `embedding_worker` (tokeniser, DataLoader, native encoder, semantic
    chunking, second pass, numpy writer) -> files on disk, through `get_encoder({'name': 'auto', ...})` on
    a local HF checkpoint directory (E1).  Rate = encoder rows (pass-1 buffers + final chunks) / wall
    seconds of the whole call, second (warm-encoder) call, max over ranks."""
    import numpy as np

    from distllm_b200.distributed_embedding import embedding_worker

    out = {}
    with tempfile.TemporaryDirectory(prefix=f'b2e_worker{rank}_') as tmp:
        tmp = Path(tmp)
        ckpt = workloads.write_bert_checkpoint(tmp / 'ckpt')
        n_docs, n_sent = 400, 30
        docs = workloads.write_semantic_docs(tmp / 'docs.jsonl', n_docs, n_sent, BERT_BASE['vocab_size'],
                                             seed=1000 + rank)
        kw = worker_kwargs(ckpt, batch=BATCH, dataset='jsonl_chunk', embedder='semantic_chunk', workers=0)
        secs, rows = [], 0
        for rep in range(2):
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            embedding_worker(docs, tmp / f'out{rep}', **kw)
            secs.append(time.perf_counter() - t0)
            rows = n_docs * n_sent + int(np.load(next((tmp / f'out{rep}').glob('*/embeddings.npy'))).shape[0])
        sec = reduce_max(secs[1])
        out['e2e_worker'] = {
            'workload': f'{n_docs} synthetic documents x {n_sent} sentences per GPU -> jsonl_chunk (buffer_size 4, '
                        '~512 tokens per buffer after truncation) -> pass 1 -> semantic split -> pass 2 -> numpy '
                        'writer; auto encoder from a local HF checkpoint dir; batch_size = chunk_batch_size = 512',
            'value': world * rows / sec, 'unit': 'encoder rows/s (512-token chunks)', 'seconds': sec,
            'rows_per_gpu': rows, 'api': 'distllm_b200.distributed_embedding.embedding_worker',
            'includes': 'file read, sentence split, tokeniser, H2D, encoder, split, pass 2, D2H, writer'}
        if do_c1:
            c1 = workloads.write_token_rows(tmp / 'c1.jsonl', 1000, 128, BERT_BASE['vocab_size'], seed=1)
            kw1 = worker_kwargs(ckpt, batch=8, workers=0)
            t = []
            for rep in range(2):
                torch.cuda.synchronize(device)
                t0 = time.perf_counter()
                embedding_worker(c1, tmp / f'c1out{rep}', **kw1)
                t.append(time.perf_counter() - t0)
            out['c1'] = {'workload': 'C1: 1 000 x 128-token chunks, mean pooler, batch_size=8, jsonl + full_sequence, '
                                     'through embedding_worker (second call, warm encoder)',
                         'value': 1000 / t[1], 'unit': 'chunks/s', 'seconds': t[1]}
    return out


def cpu_baseline_leg(device) -> dict:
    """The unmodified reference in a CPU-only subprocess on a bounded sample, then this repository's worker
    on the SAME checkpoint directory and file: the baseline number and the parity of the two outputs."""
    import numpy as np

    n_chunks = 64   # ~10-15 s of CPU work on 16 threads
    with tempfile.TemporaryDirectory(prefix='b2e_cpu_') as tmp:
        tmp = Path(tmp)
        if not reference_available():
            sec, n = cpu_oracle_run(n_chunks, 8)
            return {'value': n / sec, 'unit': 'chunks/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                    'sample': f'{n} chunks of {SEQ} tokens, batch 8, fp32 torch CPU oracle ({sec:.1f} s); '
                              'oracle/_ref absent'}
        ckpt = workloads.write_bert_checkpoint(tmp / 'ckpt')
        sample = workloads.write_token_rows(tmp / 'sample.jsonl', n_chunks, SEQ, BERT_BASE['vocab_size'], seed=123)
        cmd = [sys.executable, str(REPO / 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
               '--sample-chunks', str(n_chunks), '--checkpoint', str(ckpt), '--sample-file', str(sample),
               '--json-out', str(tmp / 'ref.json'), '--embeddings-out', str(tmp / 'ref_emb.npy'), '--no-c1']
        env = {k: v for k, v in os.environ.items()
               if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT')}
        proc = subprocess.run(cmd, env=env, capture_output=True, text=True, check=False)
        if proc.returncode != 0 or not (tmp / 'ref.json').exists():
            return {'value': None, 'kind': 'reference', 'error': proc.stderr[-600:]}
        ref = json.loads((tmp / 'ref.json').read_text())
        base = dict(ref['cpu_baseline'])
        # parity at config size against the reference's own output: same checkpoint, same file, batch 8
        from distllm_b200.distributed_embedding import embedding_worker

        embedding_worker(sample, tmp / 'ours', **worker_kwargs(ckpt, batch=8, workers=0))
        ours = np.load(next((tmp / 'ours').glob('*/embeddings.npy'))).astype(np.float64)
        theirs = np.load(tmp / 'ref_emb.npy').astype(np.float64)
        cos = (ours * theirs).sum(-1) / (np.linalg.norm(ours, axis=-1) * np.linalg.norm(theirs, axis=-1))
        base['parity_vs_reference'] = {'rows': int(len(cos)), 'min_cosine': float(cos.min()),
                                       'mean_cosine': float(cos.mean()), 'tolerance': '>= 1 - 1e-3 (north_star)',
                                       'what': 'embedding_worker output of this repository vs the unmodified '
                                               'reference on the same HF checkpoint dir and jsonl file '
                                               '(BERT-base shape, 64 chunks x 512 tokens, batch 8, mean pooler)'}
        return base


def dump_outputs(out_dir: Path, suffix: str, **arrays: torch.Tensor) -> None:
    """``--dump-outputs``: what the timed path handed back in its last step, one float32 ``.npy`` per array
    (1.5 MB per rank), so that two builds can be compared output for output on the same seeded inputs."""
    import numpy as np

    out_dir.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(out_dir / f'{name}{suffix}.npy', t.float().cpu().numpy())


def run_native(args) -> None:
    import torch.distributed as dist
    from transformers import BertConfig

    from distllm_b200 import _native as nv
    from distllm_b200.build import build_native
    from distllm_b200.embed.encoders.native import NativeBertEncoder
    from distllm_b200.embed.encoders.weights import random_bert_state_dict
    from distllm_b200.sharding import all_gather_rows
    from distllm_b200.sharding import partition_host_threads

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    partition_host_threads()   # each rank its share of the host cores (the product's torchrun driver does the same)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl native needs a B200; there is no CPU fallback')
    build_native()
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        # NCCL_DEBUG is left as the caller set it (the driver reads NCCL's own rank lines); whatever NCCL
        # prints to fd 1 lands on stderr through the redirection made in main(), never in the JSON line
        dist.init_process_group('nccl', device_id=device)

    def reduce_max(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sync_all() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    peaks, peak_src = load_peaks()
    cfg = BertConfig(**BERT_BASE)
    sd = random_bert_state_dict(cfg, seed=0, device=device)
    enc = NativeBertEncoder(cfg, sd, device=device)
    enc_storage = enc.storage   # 'bf16': the BERT family runs the bfloat16 build (fp32 accumulate / statistics)
    del sd
    hidden = BERT_BASE['hidden_size']
    steps, warm = args.steps, max(args.warmup, 3)

    # distinct synthetic ids per step and rank (the shard of the chunk stream this rank owns)
    n_distinct = min(steps, 4)
    host = [synthetic_batch(BATCH, SEQ, BERT_BASE['vocab_size'], seed=1000 * rank + i) for i in range(n_distinct)]
    dev = [tuple(t.to(device) for t in b) for b in host]
    pooled = torch.empty((steps * BATCH, hidden), dtype=torch.float32, device=device)
    last_dist = [None]

    def step(i: int) -> None:
        ids, mask, types = dev[i % n_distinct]
        out = pooled[i * BATCH:(i + 1) * BATCH]
        enc.encode_pooled(ids, mask, types, nv.POOL_MEAN_REF, False, out=out)
        last_dist[0] = nv.adjacent_cosine_dist(out)

    for i in range(warm):
        step(i % steps)
    if world > 1:
        all_gather_rows(pooled[:BATCH])  # warm the communicator
    sync_all()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for i in range(steps):
        step(i)
    gathered = all_gather_rows(pooled)  # the single collective of the run
    e1.record()
    sync_all()
    elapsed_s = reduce_max(e0.elapsed_time(e1)) * 1e-3
    clocks = sampler.stop() if rank == 0 else None
    assert gathered.shape[0] == world * steps * BATCH
    del gathered
    value = world * steps * BATCH / elapsed_s
    if args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), '' if world == 1 else f'_rank{rank}',
                     embeddings=pooled[(steps - 1) * BATCH:], adjacent_cosine_dist=last_dist[0])

    # ---- end to end through the C-ABI host-buffer call: H2D + compute + D2H inside the timing, and at
    # N > 1 the all-gather of the ranks' results (uploaded again: the user-facing result lives on the host)
    e2e_steps = min(steps, 8)
    h_ids = torch.cat([host[i % n_distinct][0] for i in range(e2e_steps)]).pin_memory()
    h_mask = torch.cat([host[i % n_distinct][1] for i in range(e2e_steps)]).pin_memory()
    h_types = torch.cat([host[i % n_distinct][2] for i in range(e2e_steps)]).pin_memory()
    h_out = torch.empty((e2e_steps * BATCH, hidden), dtype=torch.float32).pin_memory()
    enc.embed_host(h_ids[:BATCH], h_mask[:BATCH], h_types[:BATCH], BATCH, nv.POOL_MEAN_REF, False,
                   out=h_out[:BATCH])  # warm-up
    sync_all()
    t0 = time.perf_counter()
    enc.embed_host(h_ids, h_mask, h_types, BATCH, nv.POOL_MEAN_REF, False, out=h_out)
    e2e_gather_rows = 0
    if world > 1:
        full = all_gather_rows(h_out.to(device, non_blocking=True))
        e2e_gather_rows = int(full.shape[0])
        torch.cuda.synchronize(device)
    e2e_s = reduce_max(time.perf_counter() - t0)
    e2e_value = world * e2e_steps * BATCH / e2e_s
    same = torch.equal(h_out[:BATCH].to(device), pooled[:BATCH]) if n_distinct >= 1 else True
    del h_ids, h_mask, h_types

    extra: dict = {}
    # ---- ragged batches: lengths ~ U{64..512}, same batch of 512 rows (padded keys are skipped by the
    # attention kernel; padded query rows still cost GEMM / LayerNorm work -- DESIGN 8.4)
    r_ids, r_mask, r_types = (t.to(device) for t in synthetic_batch(BATCH, SEQ, BERT_BASE['vocab_size'],
                                                                     seed=77 + rank, ragged=(64, SEQ)))
    r_out = torch.empty((BATCH, hidden), dtype=torch.float32, device=device)
    r_ms = reduce_max(timed_steps(lambda: enc.encode_pooled(r_ids, r_mask, r_types, nv.POOL_MEAN_REF, False, out=r_out),
                                  5, 2, device))
    tokens = int(r_mask.sum().item())
    extra['ragged'] = {'workload': 'C2 model, batch of 512 rows padded to 512, lengths ~ U{64..512} (first row full)',
                       'value': world * BATCH / (r_ms * 1e-3), 'unit': 'chunks/s', 'ms_per_step': r_ms,
                       'attended_tokens_per_step': tokens, 'padded_tokens_per_step': BATCH * SEQ,
                       'attended_tokens_per_s': world * tokens / (r_ms * 1e-3)}
    del r_ids, r_mask, r_types, r_out

    dom = time_dominant_kernel(device, peaks) if rank == 0 else None
    if rank == 0 and world == 1 and not args.no_extras:
        extra['storage_ab'] = storage_ab(device)

    if world > 1:
        # ---- C4-sized tail: >= 2 M pooled rows per rank through the one all-gather (30.7 GB at 10 M x 768 fp32)
        rows = 2_000_000
        big = pooled[:BATCH].repeat((rows + BATCH - 1) // BATCH, 1)[:rows].contiguous()
        sync_all()
        t0 = time.perf_counter()
        full = all_gather_rows(big)
        torch.cuda.synchronize(device)
        sec = reduce_max(time.perf_counter() - t0)
        nbytes = full.numel() * 4
        extra['c4_gather'] = {'rows_per_rank': rows, 'rows_gathered': int(full.shape[0]), 'seconds': sec,
                              'bytes_received_per_gpu': nbytes * (world - 1) // world,
                              'gb_per_s_per_gpu': nbytes * (world - 1) / world / sec / 1e9,
                              'what': 'one all_gather_rows of [2 M, 768] fp32 per rank (counts exchange + '
                                      'all_gather_into_tensor), wall clock, max over ranks'}
        del big, full
        torch.cuda.empty_cache()

    enc.close()
    del enc, pooled, dev
    torch.cuda.empty_cache()
    if not args.no_extras:
        extra['c5_esm2_650m'] = extra_esm2(device, peaks, reduce_max)
        extra['c5_esm2_650m']['value'] = world * extra['c5_esm2_650m']['value_per_gpu']
        extra['c3_mistral7b'] = extra_mistral(device, peaks, reduce_max)
        extra['c3_mistral7b']['value'] = world * extra['c3_mistral7b']['value_per_gpu']
        extra.update(extra_worker(device, rank, world, reduce_max, do_c1=(world == 1)))
        if rank == 0:
            extra['retrieval'] = extra_retrieval(device, peaks)

    if rank == 0:
        fpc = flops_per_chunk(BERT_BASE, SEQ)
        step_tf = (value / world) * fpc / 1e12
        # top level: the dominant kernel against the burst peak (timed alone); whole_step: all 94
        # launches of one step against the sustained peak
        roof = {'bound': 'tensor', 'achieved': dom['achieved'], 'peak': dom['peak'], 'unit': 'TFLOP/s',
                'frac': dom['frac'], 'traffic': ncu_traffic_bytes(), 'kernel': dom['name'],
                'flops_per_launch': dom['flops_per_launch'], 'ms_per_launch': dom['ms_per_launch'],
                'peak_source': f'{peak_src} burst 16-bit (bf16 cuBLAS) tensor peak (kernel timed alone)',
                'whole_step': {'achieved': step_tf, 'peak': peaks['bf16_tflops_sustained'],
                               'frac': step_tf / peaks['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                               'flops_per_chunk': fpc,
                               'peak_source': f'{peak_src} sustained 16-bit (bf16 cuBLAS) tensor peak (whole step, per GPU)'}}
        cpu_base = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_base = cpu_baseline_leg(device)
        line = {
            'metric': METRIC, 'value': value, 'unit': 'chunks/s', 'n_gpus': world,
            'steps': steps, 'warmup': warm, 'ms_per_step': 1e3 * elapsed_s / steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': enc_storage, 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'global_batch': BATCH * world, 'seq_len': SEQ,
                       'parallelism': f'dp{world}: chunks sharded by rank, one all-gather of the pooled matrix',
                       'l2': 'per-step activations (~4 GB) exceed the 126 MB L2; no explicit flush needed'},
            'e2e': {'value': e2e_value, 'unit': 'chunks/s', 'h2d_bytes_per_step': 3 * BATCH * SEQ * 8,
                    'd2h_bytes_per_step': BATCH * hidden * 4, 'steps': e2e_steps,
                    'api': 'b2e_embed_host (C ABI, pinned host buffers)' + (
                        ' + one all-gather of the result matrices' if world > 1 else ''),
                    'all_gather_rows': e2e_gather_rows, 'matches_device_path': bool(same)},
            'gpu_launches': launches_per_step(BERT_BASE) * steps,
            'clocks': clocks, 'roofline': roof, 'cpu_baseline': cpu_base, 'extra': extra,
        }
        emit(line, args.json_out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', choices=['native', 'reference'], default='native')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the CPU reference timing leg')
    ap.add_argument('--no-extras', action='store_true', help='skip the C3 / C5 / worker extras (profiling runs)')
    # reference arm knobs (the native arm's cpu_baseline leg drives them)
    ap.add_argument('--sample-chunks', type=int, default=8, help='chunks per reference step (bounded sample)')
    ap.add_argument('--data-workers', type=int, default=4, help="DataLoader workers (the reference's default: 4)")
    ap.add_argument('--checkpoint', default=None, help='existing HF checkpoint directory to embed with')
    ap.add_argument('--sample-file', default=None, help='existing jsonl file to use as the step input')
    ap.add_argument('--json-out', default=None, help='also write the JSON line to this file')
    ap.add_argument('--embeddings-out', default=None, help='copy the last step embeddings.npy here')
    ap.add_argument('--no-c1', dest='with_c1', action='store_false', help='skip the C1 (1000 x 128-token) run')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the last timed step's pooled embeddings and adjacent-cosine distances to "
                         'DIR/<name>.npy (native arm)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'native':
        ap.error('--dump-outputs applies to the native arm')
    # stdout carries exactly one JSON line: everything libraries write to fd 1 while the benchmark
    # runs (NCCL's version banner, progress bars) is sent to stderr; emit() writes to the saved fd
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_native(args)


_JSON_FD = None


def emit(line: dict, also_to: str | None = None) -> None:
    payload = (json.dumps(line) + '\n').encode()
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, payload)
    if also_to:
        Path(also_to).write_bytes(payload)


if __name__ == '__main__':
    main()
