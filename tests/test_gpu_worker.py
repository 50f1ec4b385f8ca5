"""-m gpu: the plugin-level entry points on a B200, from files on disk to files on disk.

W1 `embedding_worker`, E1 `get_encoder({'name': 'auto' | 'esm2', ...}, register=True)` on local HF checkpoint
directories (``save_pretrained``), the typer CLI and the torchrun driver -- compared with the outputs the
UNMODIFIED reference produced for the same checkpoints and texts (tests/golden/*.npz, written by
oracle/make_golden.py from the unmodified reference copied into oracle/_ref).
"""

from __future__ import annotations

import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import REPO
from conftest import cosine_rows

pytestmark = pytest.mark.gpu
COS_TOL = 1e-3


def worker_kwargs(ckpt: Path, encoder: str = 'auto', dataset: str = 'jsonl', pooler: str = 'mean',
                  writer: str = 'numpy', batch: int = 4, **dataset_extra) -> dict:
    enc = {'name': encoder, 'pretrained_model_name_or_path': str(ckpt), 'half_precision': False}
    if encoder == 'auto':
        enc['quantization'] = False
    return dict(
        dataset_kwargs={'name': dataset, 'batch_size': batch, 'num_data_workers': 0, 'pin_memory': True,
                        **dataset_extra},
        encoder_kwargs=enc,
        pooler_kwargs={'name': pooler},
        embedder_kwargs={'name': 'full_sequence'},
        writer_kwargs={'name': writer},
    )


@pytest.fixture(scope='module')
def bert_ckpt(tmp_path_factory):
    from oracle.make_golden import tiny_bert_texts
    from oracle.make_golden import write_tiny_bert_checkpoint

    root = tmp_path_factory.mktemp('bert')
    write_tiny_bert_checkpoint(root / 'ckpt')
    texts = tiny_bert_texts()
    (root / 'in').mkdir()
    (root / 'in' / 'texts.jsonl').write_text('\n'.join(json.dumps({'text': t}) for t in texts) + '\n')
    return root, texts


def read_single_output(out_dir: Path) -> Path:
    dirs = [p for p in out_dir.iterdir() if p.is_dir()]
    assert len(dirs) == 1, dirs
    return dirs[0]


def test_embedding_worker_bert_checkpoint_dir_matches_reference(bert_ckpt, bert_golden, capsys):
    """HF checkpoint dir -> registry warm start -> tokenizer/DataLoader -> native encoder -> numpy writer,
    against the reference's compute_embeddings output for the same 14 texts in batches of 4."""
    from distllm_b200.distributed_embedding import embedding_worker
    from distllm_b200.embed import get_encoder
    from distllm_b200.registry import registry

    root, texts = bert_ckpt
    kw = worker_kwargs(root / 'ckpt')
    embedding_worker(root / 'in' / 'texts.jsonl', root / 'out_np', **kw)
    timers = [line for line in capsys.readouterr().out.splitlines() if line.startswith('[timer]')]
    assert [t.split('] [')[1].split()[0] for t in timers] == [
        'loaded-encoder', 'loaded-dataset', 'computed-embeddings', 'wrote-embeddings', 'finished-embedding']
    d = read_single_output(root / 'out_np')
    emb = np.load(d / 'embeddings.npy')
    assert emb.dtype == np.float32 and emb.shape == bert_golden['pooled/mean'].shape
    assert np.load(d / 'text.npy').tolist() == texts
    cos = cosine_rows(emb, bert_golden['pooled/mean'])
    assert cos.min() > 1 - COS_TOL, cos
    # warm start: the same kwargs hand back the SAME encoder object (weights + native workspace kept)
    enc1 = get_encoder(kw['encoder_kwargs'], register=True)
    assert get_encoder(kw['encoder_kwargs'], register=True) is enc1
    assert enc1.tokenizer.model_max_length == 64 and enc1.embedding_size == 256
    # the tokenizer path produced the reference's token batches
    batch = enc1.tokenizer(texts[:4], padding=True, truncation=True, return_tensors='pt')
    assert np.array_equal(batch['input_ids'].numpy(), bert_golden['batch0/input_ids'])
    # last_token pooler + huggingface writer through the same worker
    kw2 = worker_kwargs(root / 'ckpt', pooler='last_token', writer='huggingface')
    embedding_worker(root / 'in' / 'texts.jsonl', root / 'out_hf', **kw2)
    import datasets

    table = datasets.Dataset.load_from_disk(str(read_single_output(root / 'out_hf')))
    assert table.column_names[:2] == ['text', 'embeddings'] and table['text'] == texts
    cos = cosine_rows(np.asarray(table['embeddings'], dtype=np.float32), bert_golden['pooled/last_token'])
    assert cos.min() > 1 - COS_TOL, cos
    registry.clear()


def test_embedding_worker_esm2_checkpoint_dir_matches_reference(tmp_path, esm_golden):
    """`esm2` encoder from a checkpoint dir (EsmForMaskedLM weights, EsmTokenizer) through the worker."""
    from distllm_b200.distributed_embedding import embedding_worker
    from distllm_b200.registry import registry
    from oracle.make_golden import tiny_esm_seqs
    from oracle.make_golden import write_tiny_esm_checkpoint

    write_tiny_esm_checkpoint(tmp_path / 'ckpt')
    seqs = tiny_esm_seqs()
    (tmp_path / 'seqs.txt').write_text('header\n' + '\n'.join(seqs) + '\n')
    kw = worker_kwargs(tmp_path / 'ckpt', encoder='esm2', dataset='sequence_per_line')
    embedding_worker(tmp_path / 'seqs.txt', tmp_path / 'out', **kw)
    emb = np.load(read_single_output(tmp_path / 'out') / 'embeddings.npy')
    ref = esm_golden['pooled/mean']
    assert emb.shape == ref.shape
    live = np.linalg.norm(ref, axis=-1) > 0     # the 1-residue row pools to zeros on both sides
    assert not emb[~live].any()
    cos = cosine_rows(emb[live], ref[live])
    assert cos.min() > 1 - COS_TOL, cos
    registry.clear()


def test_embedding_worker_mistral_checkpoint_dir_matches_reference(tmp_path, mistral_golden):
    """`auto` encoder on a MistralModel checkpoint dir (q/k/v/o, gate/up/down re-laid out by weights.py)."""
    from distllm_b200.distributed_embedding import embedding_worker
    from distllm_b200.registry import registry
    from oracle.make_golden import tiny_mistral_texts
    from oracle.make_golden import write_tiny_mistral_checkpoint

    write_tiny_mistral_checkpoint(tmp_path / 'ckpt')
    texts = tiny_mistral_texts()
    (tmp_path / 't.jsonl').write_text('\n'.join(json.dumps({'text': t}) for t in texts) + '\n')
    kw = worker_kwargs(tmp_path / 'ckpt', pooler='last_token')
    embedding_worker(tmp_path / 't.jsonl', tmp_path / 'out', **kw)
    emb = np.load(read_single_output(tmp_path / 'out') / 'embeddings.npy')
    cos = cosine_rows(emb, mistral_golden['full/right/pooled/last_token'])
    assert cos.min() > 1 - COS_TOL, cos
    registry.clear()


def test_cli_embed_and_merge_end_to_end(bert_ckpt, bert_golden, tmp_path):
    """`python -m distllm_b200.cli embed ...` with the reference's flag spellings (distllm/cli.py:14-192),
    two input files, then `merge` (cli.py:195-245)."""
    root, texts = bert_ckpt
    data = tmp_path / 'data'
    data.mkdir()
    (data / 'a.jsonl').write_text('\n'.join(json.dumps({'text': t}) for t in texts[:8]) + '\n')
    (data / 'b.jsonl').write_text('\n'.join(json.dumps({'text': t}) for t in texts[8:]) + '\n')
    env = {**os.environ, 'PYTHONPATH': str(REPO)}
    cmd = [sys.executable, '-m', 'distllm_b200.cli', 'embed', '--encoder_name', 'auto', '-m', str(root / 'ckpt'),
           '-d', str(data), '-de', 'jsonl', '-o', str(tmp_path / 'emb'), '--dataset_name', 'jsonl', '-b', '4',
           '--pooler_name', 'mean', '--embedder_name', 'full_sequence', '--writer_name', 'numpy', '--eval_mode']
    proc = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600, check=False)
    assert proc.returncode == 0, proc.stderr[-2000:]
    assert proc.stdout.count('[timer] [computed-embeddings') == 2
    proc = subprocess.run([sys.executable, '-m', 'distllm_b200.cli', 'merge', '--writer_name', 'numpy',
                           '-d', str(tmp_path / 'emb'), '-o', str(tmp_path / 'merged')],
                          env=env, capture_output=True, text=True, timeout=600, check=False)
    assert proc.returncode == 0, proc.stderr[-2000:]
    merged_text = np.load(tmp_path / 'merged' / 'text.npy').tolist()
    emb = np.load(tmp_path / 'merged' / 'embeddings.npy')
    assert sorted(merged_text) == sorted(texts)
    # rows 0..7 are two full reference batches; the order of the two files is the writer directories' order
    ref = {t: r for t, r in zip(texts, bert_golden['pooled/mean'])}
    got = {t: r for t, r in zip(merged_text, emb)}
    first8 = np.stack([got[t] for t in texts[:8]])
    cos = cosine_rows(first8, np.stack([ref[t] for t in texts[:8]]))
    assert cos.min() > 1 - COS_TOL, cos


def test_torchrun_driver_two_ranks_gather(bert_ckpt, bert_golden, tmp_path):
    """`torchrun -m distllm_b200.distributed_embedding --config ... --gather` with 2 ranks: documents (jsonl
    lines of ONE input file) sharded by rank, device-resident rows all-gathered, rank 0 writes the matrix in
    document order.  Both ranks share the box's single GPU, so the collective runs on gloo here (NCCL refuses
    two ranks on one device); the NCCL path is what bench.py --gpus N exercises."""
    import socket

    root, texts = bert_ckpt
    cfg = {
        'input_dir': str(root / 'in'), 'output_dir': str(tmp_path / 'run'), 'glob_patterns': ['*.jsonl'],
        'dataset_config': {'name': 'jsonl', 'batch_size': 4, 'num_data_workers': 0},
        'encoder_config': {'name': 'auto', 'pretrained_model_name_or_path': str(root / 'ckpt'),
                           'quantization': False},
        'pooler_config': {'name': 'last_token'},
        'embedder_config': {'name': 'full_sequence'},
        'writer_config': {'name': 'numpy'},
    }
    import yaml

    (tmp_path / 'cfg.yaml').write_text(yaml.safe_dump(cfg))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    env = {**os.environ, 'PYTHONPATH': str(REPO), 'B2E_DIST_BACKEND': 'gloo'}
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', str(port),
           '-m', 'distllm_b200.distributed_embedding', '--config', str(tmp_path / 'cfg.yaml'), '--gather']
    proc = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900, check=False)
    assert proc.returncode == 0, (proc.stdout[-1500:], proc.stderr[-3000:])
    full = np.load(tmp_path / 'run' / 'embeddings_all.npy')
    ref = bert_golden['pooled/last_token']     # last-token pooling does not depend on batch composition
    assert full.shape == ref.shape
    cos = cosine_rows(full, ref)
    assert cos.min() > 1 - COS_TOL, cos
    # each rank wrote its own document range: 7 + 7 rows, texts in document order
    parts = sorted((tmp_path / 'run' / 'embeddings').iterdir())
    got_texts = sorted(t for p in parts for t in np.load(p / 'text.npy').tolist())
    assert got_texts == sorted(texts) and len(parts) == 2
    assert not (tmp_path / 'run' / '.shards' / 'rank0').exists()


def test_embedding_worker_semantic_chunk_matches_reference_worker(bert_ckpt, tmp_path):
    """File in -> files out through jsonl_chunk + semantic_chunk + mean + numpy writer, against what the
    reference's own `embedding_worker` wrote for the same documents (tests/golden/worker_golden.npz):
    the chunk texts (the discrete split) must be identical, the chunk embeddings within 1e-3 cosine."""
    from distllm_b200.distributed_embedding import embedding_worker
    from distllm_b200.registry import registry
    from oracle.make_golden import WORKER_DATASET
    from oracle.make_golden import WORKER_EMBEDDER
    from oracle.make_golden import worker_docs

    golden = np.load(REPO / 'tests' / 'golden' / 'worker_golden.npz')
    root, _ = bert_ckpt
    f = tmp_path / 'docs.jsonl'
    f.write_text('\n'.join(json.dumps(d) for d in worker_docs()))
    embedding_worker(
        f, tmp_path / 'out',
        dataset_kwargs={**WORKER_DATASET, 'sentence_splitter': 'regex'},   # the splitter the golden was made with
        encoder_kwargs={'name': 'auto', 'pretrained_model_name_or_path': str(root / 'ckpt'), 'quantization': False},
        pooler_kwargs={'name': 'mean'},
        embedder_kwargs=dict(WORKER_EMBEDDER),
        writer_kwargs={'name': 'numpy'},
    )
    out = read_single_output(tmp_path / 'out')
    assert np.load(out / 'text.npy').tolist() == golden['text'].tolist()
    meta = np.load(out / 'metadata.npy', allow_pickle=True)
    assert [m['path'] for m in meta] == golden['paths'].tolist() and all('sentence' not in m for m in meta)
    cos = cosine_rows(np.load(out / 'embeddings.npy'), golden['embeddings'])
    assert cos.min() > 1 - COS_TOL, cos
    registry.clear()


def test_embedding_worker_modernbert_checkpoint_dir_matches_reference(tmp_path, modernbert_golden):
    """`auto` encoder on a ModernBertModel checkpoint dir (the family of the reference's
    examples/embed/workstation/modernbert_semchunk.yaml) through the worker, normalised mean embeddings."""
    from distllm_b200.distributed_embedding import embedding_worker
    from distllm_b200.registry import registry
    from oracle.make_golden import tiny_modernbert_texts
    from oracle.make_golden import write_tiny_modernbert_checkpoint

    write_tiny_modernbert_checkpoint(tmp_path / 'ckpt')
    texts = tiny_modernbert_texts()
    (tmp_path / 't.jsonl').write_text('\n'.join(json.dumps({'text': t}) for t in texts) + '\n')
    kw = worker_kwargs(tmp_path / 'ckpt')
    kw['embedder_kwargs'] = {'name': 'full_sequence', 'normalize_embeddings': True}
    embedding_worker(tmp_path / 't.jsonl', tmp_path / 'out', **kw)
    emb = np.load(read_single_output(tmp_path / 'out') / 'embeddings.npy')
    ref = modernbert_golden['pooled/mean_normalized']
    live = np.linalg.norm(ref, axis=-1) > 0
    assert not emb[~live].any()
    cos = cosine_rows(emb[live], ref[live])
    assert cos.min() > 1 - COS_TOL, cos
    registry.clear()


def test_auto_encoder_quantization_true_runs_nf4_weights(bert_ckpt):
    """`quantization=True` (the reference's YAML default, auto.py:31,44-56): the native GEMMs run on
    dequant(NF4(W)).  Checked against the oracle forward on the SAME round-tripped weights (cosine) and against
    the unquantised model (must differ: NF4 changes every Linear weight by ~9 %)."""
    import torch
    from transformers import BertConfig

    from distllm_b200.embed import get_encoder
    from distllm_b200.embed.encoders.nf4 import quantize_state_dict_nf4
    from distllm_b200.embed.encoders.weights import random_bert_state_dict
    from oracle import bert as obert
    from oracle.make_golden import TINY
    from oracle.make_golden import TINY_SEED

    root, texts = bert_ckpt
    enc_q = get_encoder({'name': 'auto', 'pretrained_model_name_or_path': str(root / 'ckpt'), 'quantization': True})
    batch = enc_q.tokenizer(texts[:4], padding=True, truncation=True, return_tensors='pt')
    on_device = enc_q.tokenizer(texts[:4], padding=True, truncation=True, return_tensors='pt').to(enc_q.device)
    got = enc_q.encode(on_device).cpu().numpy()   # (BatchEncoding.to moves in place: `batch` stays on the host)
    cfg = BertConfig(**TINY)
    sd = random_bert_state_dict(cfg, seed=TINY_SEED, device='cpu')
    ref_q = obert.bert_forward(quantize_state_dict_nf4(sd), cfg, batch['input_ids'], batch['attention_mask'],
                               batch['token_type_ids']).numpy()
    ref_f = obert.bert_forward(sd, cfg, batch['input_ids'], batch['attention_mask'], batch['token_type_ids']).numpy()
    valid = batch['attention_mask'].bool().numpy()
    assert cosine_rows(got[valid], ref_q[valid]).min() > 1 - COS_TOL
    assert cosine_rows(got[valid], ref_f[valid]).min() < 1 - 1e-3     # quantisation is visible
    enc_q.native.close()
