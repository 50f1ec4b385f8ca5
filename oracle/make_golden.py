"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU.

Needs the reference in ``oracle/_ref``, which ``oracle/ref_shims.install_reference`` copies in first
(``DISTLLM_REFERENCE=<distllm checkout>`` picks another checkout than its default):

    python oracle/make_golden.py

What is recorded (all seeded, fp32, CPU):
  pool_golden.npz      distllm.embed.poolers.mean.average_pool / last_token.last_token_pool on ragged
                       batches (outputs + the mask after the in-place edit)
  semantic_golden.npz  distllm.embed.embedders.semantic_chunk.calculate_distances_between_buffer and
                       build_chunks on random embeddings, incl. 1- and 2-row documents
  worker_golden.npz    the reference's own embedding_worker, file in -> files out (jsonl_chunk +
                       semantic_chunk + mean + numpy writer) on the tiny BERT checkpoint
  bert_tiny_golden.npz the reference's own AutoEncoder + poolers + compute_embeddings
                       (distllm/embed/embedders/full_sequence.py:20-80) driven through a real DataLoader
                       and tokenizer on a tiny seeded BERT checkpoint: token batches, first-batch hidden
                       state, pooled embeddings (mean / mean+normalize / last_token)

TEST INFRASTRUCTURE ONLY.
"""

from __future__ import annotations

import hashlib
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
GOLDEN = REPO / 'tests' / 'golden'

TINY = dict(vocab_size=200, hidden_size=256, num_hidden_layers=2, num_attention_heads=4,
            intermediate_size=512, max_position_embeddings=64, type_vocab_size=2,
            layer_norm_eps=1e-12, hidden_act='gelu', hidden_dropout_prob=0.0,
            attention_probs_dropout_prob=0.0, initializer_range=0.05)
TINY_SEED = 1234


def weights_digest(sd: dict[str, torch.Tensor]) -> str:
    h = hashlib.sha256()
    for key in sorted(sd):
        h.update(key.encode())
        h.update(sd[key].detach().cpu().float().numpy().tobytes())
    return h.hexdigest()


def make_pool_golden() -> None:
    from distllm.embed.poolers.last_token import last_token_pool
    from distllm.embed.poolers.mean import average_pool

    g = torch.Generator().manual_seed(7)
    out = {}
    cases = {
        'ragged': [20, 5, 1, 2, 11, 11, 19, 0],       # includes len 0 (index -1 wraps), 1, 2, dup lens
        'full': [12, 12, 12],
        'single': [9],
        'left_padded_like': [7, 16, 16],               # last column set for some rows only
    }
    for name, lens in cases.items():
        s = max(max(lens), 2)
        b = len(lens)
        emb = torch.randn(b, s, 256, generator=g)
        mask = (torch.arange(s)[None, :] < torch.tensor(lens)[:, None]).long()
        m1 = mask.clone()
        pooled = average_pool(emb, m1)
        out[f'{name}/emb'] = emb.numpy()
        out[f'{name}/mask'] = mask.numpy()
        out[f'{name}/mean'] = pooled.numpy()
        out[f'{name}/mask_after'] = m1.numpy()
        if min(lens) > 0:
            out[f'{name}/last'] = last_token_pool(emb, mask.clone()).numpy()
    # left padding: every row ends attended -> column S-1 branch of last_token_pool
    emb = torch.randn(4, 10, 256, generator=g)
    mask = (torch.arange(10)[None, :] >= torch.tensor([0, 3, 7, 9])[:, None]).long()
    out['leftpad/emb'] = emb.numpy()
    out['leftpad/mask'] = mask.numpy()
    out['leftpad/last'] = last_token_pool(emb, mask.clone()).numpy()
    np.savez_compressed(GOLDEN / 'pool_golden.npz', **out)


def make_semantic_golden() -> None:
    from distllm.embed.embedders.semantic_chunk import build_chunks
    from distllm.embed.embedders.semantic_chunk import calculate_distances_between_buffer

    rng = np.random.default_rng(11)
    emb = rng.standard_normal((64, 256)).astype(np.float32)
    # correlated neighbours so distances spread over (0, 1)
    for i in range(1, 64):
        emb[i] = 0.6 * emb[i - 1] + rng.uniform(0.1, 1.0) * emb[i]
    doc_ranges = [(0, 25), (25, 26), (26, 28), (28, 64)]
    out = {'emb': emb, 'doc_ranges': np.array(doc_ranges)}
    for k, (lo, hi) in enumerate(doc_ranges):
        d = calculate_distances_between_buffer(emb[lo:hi])
        out[f'dist/{k}'] = d
        for pct in (50, 90, 95):
            out[f'groups/{k}/{pct}'] = np.array(build_chunks(d, pct))
    np.savez_compressed(GOLDEN / 'semantic_golden.npz', **out)


def tiny_bert_vocab() -> list[str]:
    words = [f'w{i:03d}' for i in range(TINY['vocab_size'] - 5)]
    return ['[PAD]', '[UNK]', '[CLS]', '[SEP]', '[MASK]', *words]


def tiny_bert_texts() -> list[str]:
    """The 14 texts behind bert_tiny_golden.npz (80 words -> truncated to 64 tokens)."""
    words = tiny_bert_vocab()[5:]
    rng = np.random.default_rng(5)
    lengths = [3, 17, 40, 1, 25, 25, 9, 62, 80, 12, 30, 2, 44, 7]
    return [' '.join(rng.choice(words, size=n)) for n in lengths]


def write_tiny_bert_checkpoint(ckpt_dir: Path) -> None:
    """HF checkpoint directory (config.json, weights, tokenizer files) of the tiny seeded BERT."""
    from transformers import BertConfig
    from transformers import BertModel
    from transformers import BertTokenizerFast

    from distllm_b200.embed.encoders.weights import random_bert_state_dict

    cfg = BertConfig(**TINY)
    sd = random_bert_state_dict(cfg, seed=TINY_SEED, device='cpu')
    model = BertModel(cfg)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith('pooler.') for k in missing), (missing, unexpected)
    ckpt_dir = Path(ckpt_dir)
    ckpt_dir.mkdir(parents=True, exist_ok=True)
    (ckpt_dir / 'vocab.txt').write_text('\n'.join(tiny_bert_vocab()) + '\n')
    tok = BertTokenizerFast(vocab=str(ckpt_dir / 'vocab.txt'), do_lower_case=False)
    model.eval().save_pretrained(ckpt_dir)
    tok.save_pretrained(ckpt_dir)


def make_bert_golden() -> None:
    from torch.utils.data import DataLoader
    from transformers import BertConfig
    from transformers import BertModel
    from transformers import BertTokenizerFast

    from distllm.embed.datasets.utils import DataCollator
    from distllm.embed.datasets.utils import InMemoryDataset
    from distllm.embed.embedders.full_sequence import compute_embeddings
    from distllm.embed.encoders.auto import AutoEncoder
    from distllm.embed.encoders.auto import AutoEncoderConfig
    from distllm.embed.poolers.last_token import LastTokenPooler
    from distllm.embed.poolers.last_token import LastTokenPoolerConfig
    from distllm.embed.poolers.mean import MeanPooler
    from distllm.embed.poolers.mean import MeanPoolerConfig
    from distllm_b200.embed.encoders.weights import random_bert_state_dict

    cfg = BertConfig(**TINY)
    sd = random_bert_state_dict(cfg, seed=TINY_SEED, device='cpu')
    texts = tiny_bert_texts()
    n_texts = len(texts)

    with tempfile.TemporaryDirectory() as tmp:
        tmp_path = Path(tmp)
        write_tiny_bert_checkpoint(tmp_path / 'ckpt')

        encoder = AutoEncoder(AutoEncoderConfig(
            pretrained_model_name_or_path=str(tmp_path / 'ckpt'), quantization=False, eval_mode=True))
        assert encoder.tokenizer.model_max_length == TINY['max_position_embeddings']

        def loader() -> DataLoader:
            return DataLoader(InMemoryDataset(texts), batch_size=4, num_workers=0,
                              collate_fn=DataCollator(encoder.tokenizer))

        out = {'weights_sha256': np.array(weights_digest(sd)), 'n_texts': np.array(n_texts)}
        for i, batch in enumerate(loader()):
            out[f'batch{i}/input_ids'] = batch['input_ids'].numpy()
            out[f'batch{i}/attention_mask'] = batch['attention_mask'].numpy()
            out[f'batch{i}/token_type_ids'] = batch['token_type_ids'].numpy()
            if i == 0:
                with torch.no_grad():
                    out['batch0/hidden'] = encoder.encode(batch).numpy()
        out['n_batches'] = np.array(i + 1)
        mean = MeanPooler(MeanPoolerConfig())
        last = LastTokenPooler(LastTokenPoolerConfig())
        out['pooled/mean'] = compute_embeddings(loader(), encoder, mean)
        out['pooled/mean_normalized'] = compute_embeddings(loader(), encoder, mean, normalize=True)
        out['pooled/last_token'] = compute_embeddings(loader(), encoder, last)
    np.savez_compressed(GOLDEN / 'bert_tiny_golden.npz', **out)


TINY_ESM = dict(vocab_size=33, hidden_size=256, num_hidden_layers=2, num_attention_heads=4,
                intermediate_size=512, max_position_embeddings=160, position_embedding_type='rotary',
                token_dropout=True, mask_token_id=32, pad_token_id=1, layer_norm_eps=1e-5,
                emb_layer_norm_before=False, hidden_dropout_prob=0.0,
                attention_probs_dropout_prob=0.0, initializer_range=0.05)
TINY_ESM_SEED = 4321
ESM_VOCAB = ['<cls>', '<pad>', '<eos>', '<unk>', 'L', 'A', 'G', 'V', 'S', 'E', 'R', 'T', 'I', 'D', 'P',
             'K', 'Q', 'N', 'F', 'Y', 'M', 'H', 'W', 'C', 'X', 'B', 'U', 'Z', 'O', '.', '-', '<null_1>',
             '<mask>']


def tiny_esm_seqs() -> list[str]:
    """The 10 sequences behind esm_tiny_golden.npz (200 residues -> truncated to 160 tokens)."""
    rng = np.random.default_rng(9)
    residues = list('LAGVSERTIDPKQNFYMHWC')
    lengths = [12, 150, 33, 1, 64, 64, 200, 7, 90, 41]
    seqs = [''.join(rng.choice(residues, size=n)) for n in lengths]
    seqs[2] = seqs[2][:10] + '<mask>' + seqs[2][10:20] + '<mask>' + seqs[2][20:]  # token-dropout rows
    return seqs


def write_tiny_esm_checkpoint(ckpt_dir: Path) -> None:
    from transformers import EsmConfig
    from transformers import EsmForMaskedLM
    from transformers import EsmTokenizer

    from distllm_b200.embed.encoders.weights import random_esm_state_dict

    cfg = EsmConfig(**TINY_ESM)
    sd = random_esm_state_dict(cfg, seed=TINY_ESM_SEED, device='cpu')
    model = EsmForMaskedLM(cfg)
    missing, unexpected = model.load_state_dict({'esm.' + k: v for k, v in sd.items()}, strict=False)
    assert not unexpected, unexpected
    # missing = parts the hot path never touches (LM head, contact head) and the rotary inv_freq buffers
    assert all(k.startswith(('lm_head.', 'esm.contact_head.', 'esm.embeddings.position'))
               or k.endswith('rotary_embeddings.inv_freq') for k in missing), missing
    ckpt_dir = Path(ckpt_dir)
    ckpt_dir.mkdir(parents=True, exist_ok=True)
    (ckpt_dir / 'vocab.txt').write_text('\n'.join(ESM_VOCAB) + '\n')
    tok = EsmTokenizer(str(ckpt_dir / 'vocab.txt'))
    model.eval().save_pretrained(ckpt_dir)
    tok.save_pretrained(ckpt_dir)


def make_esm_golden() -> None:
    """The reference's own Esm2Encoder (HF EsmForMaskedLM) + MeanPooler + compute_embeddings on a
    tiny seeded ESM-2 checkpoint with rotary positions and token dropout."""
    from torch.utils.data import DataLoader
    from transformers import EsmConfig
    from transformers import EsmForMaskedLM
    from transformers import EsmTokenizer

    from distllm.embed.datasets.utils import DataCollator
    from distllm.embed.datasets.utils import InMemoryDataset
    from distllm.embed.embedders.full_sequence import compute_embeddings
    from distllm.embed.encoders.esm2 import Esm2Encoder
    from distllm.embed.encoders.esm2 import Esm2EncoderConfig
    from distllm.embed.poolers.mean import MeanPooler
    from distllm.embed.poolers.mean import MeanPoolerConfig
    from distllm_b200.embed.encoders.weights import random_esm_state_dict

    cfg = EsmConfig(**TINY_ESM)
    sd = random_esm_state_dict(cfg, seed=TINY_ESM_SEED, device='cpu')
    seqs = tiny_esm_seqs()

    with tempfile.TemporaryDirectory() as tmp:
        tmp_path = Path(tmp)
        write_tiny_esm_checkpoint(tmp_path / 'ckpt')
        encoder = Esm2Encoder(Esm2EncoderConfig(
            pretrained_model_name_or_path=str(tmp_path / 'ckpt'), half_precision=False))
        assert encoder.tokenizer.model_max_length == TINY_ESM['max_position_embeddings']

        def loader() -> DataLoader:
            return DataLoader(InMemoryDataset(seqs), batch_size=4, num_workers=0,
                              collate_fn=DataCollator(encoder.tokenizer))

        out = {'weights_sha256': np.array(weights_digest(sd)), 'n_texts': np.array(len(seqs))}
        for i, batch in enumerate(loader()):
            out[f'batch{i}/input_ids'] = batch['input_ids'].numpy()
            out[f'batch{i}/attention_mask'] = batch['attention_mask'].numpy()
            if i == 0:
                with torch.no_grad():
                    out['batch0/hidden'] = encoder.encode(batch).numpy()
        out['n_batches'] = np.array(i + 1)
        out['pooled/mean'] = compute_embeddings(loader(), encoder, MeanPooler(MeanPoolerConfig()))
    np.savez_compressed(GOLDEN / 'esm_tiny_golden.npz', **out)


TINY_MISTRAL = dict(vocab_size=320, hidden_size=512, num_hidden_layers=2, num_attention_heads=4,
                    num_key_value_heads=2, head_dim=128, intermediate_size=768,
                    max_position_embeddings=320, rms_norm_eps=1e-5, hidden_act='silu',
                    sliding_window=None, attention_dropout=0.0, initializer_range=0.05,
                    pad_token_id=0, bos_token_id=1, eos_token_id=2)
TINY_MISTRAL_SEED = 2468
TINY_MISTRAL_WINDOW = 80   # second variant: same weights, sliding-window attention


def tiny_mistral_texts() -> list[str]:
    """The 12 texts behind mistral_tiny_golden.npz (400 words -> truncated to 320 tokens)."""
    words = [f'w{i:03d}' for i in range(TINY_MISTRAL['vocab_size'] - 4)]
    rng = np.random.default_rng(21)
    lengths = [5, 150, 33, 1, 64, 63, 400, 7, 127, 128, 200, 90]
    return [' '.join(rng.choice(words, size=n)) for n in lengths]


def write_tiny_mistral_checkpoint(ckpt_dir: Path, window: int | None = None) -> None:
    from tokenizers import Tokenizer
    from tokenizers.models import WordLevel
    from tokenizers.pre_tokenizers import Whitespace
    from tokenizers.processors import TemplateProcessing
    from transformers import MistralConfig
    from transformers import MistralModel
    from transformers import PreTrainedTokenizerFast

    from distllm_b200.embed.encoders.weights import random_mistral_state_dict

    words = [f'w{i:03d}' for i in range(TINY_MISTRAL['vocab_size'] - 4)]
    vocab = {t: i for i, t in enumerate(['<pad>', '<s>', '</s>', '<unk>', *words])}
    cfg = MistralConfig(**{**TINY_MISTRAL, 'sliding_window': window})
    sd = random_mistral_state_dict(cfg, seed=TINY_MISTRAL_SEED, device='cpu')
    model = MistralModel(cfg)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all('rotary_emb' in k for k in missing), (missing, unexpected)
    raw = Tokenizer(WordLevel(vocab, unk_token='<unk>'))
    raw.pre_tokenizer = Whitespace()
    raw.post_processor = TemplateProcessing(single='<s> $A', special_tokens=[('<s>', 1)])
    tok = PreTrainedTokenizerFast(tokenizer_object=raw, pad_token='<pad>', bos_token='<s>',
                                  eos_token='</s>', unk_token='<unk>')
    model.eval().save_pretrained(ckpt_dir)
    tok.save_pretrained(ckpt_dir)


def make_mistral_golden() -> None:
    """The reference's AutoEncoder (HF MistralModel: grouped-query causal attention, rotary, RMSNorm,
    SwiGLU) + LastTokenPooler / MeanPooler + compute_embeddings on a tiny seeded checkpoint, with
    right- and left-padded batches, without and with a sliding window."""
    from tokenizers import Tokenizer
    from tokenizers.models import WordLevel
    from tokenizers.pre_tokenizers import Whitespace
    from tokenizers.processors import TemplateProcessing
    from torch.utils.data import DataLoader
    from transformers import MistralConfig
    from transformers import MistralModel
    from transformers import PreTrainedTokenizerFast

    from distllm.embed.datasets.utils import DataCollator
    from distllm.embed.datasets.utils import InMemoryDataset
    from distllm.embed.embedders.full_sequence import compute_embeddings
    from distllm.embed.encoders.auto import AutoEncoder
    from distllm.embed.encoders.auto import AutoEncoderConfig
    from distllm.embed.poolers.last_token import LastTokenPooler
    from distllm.embed.poolers.last_token import LastTokenPoolerConfig
    from distllm.embed.poolers.mean import MeanPooler
    from distllm.embed.poolers.mean import MeanPoolerConfig
    from distllm_b200.embed.encoders.weights import random_mistral_state_dict

    texts = tiny_mistral_texts()
    out = {'n_texts': np.array(len(texts))}

    for variant, window in (('full', None), ('window', TINY_MISTRAL_WINDOW)):
        cfg = MistralConfig(**{**TINY_MISTRAL, 'sliding_window': window})
        sd = random_mistral_state_dict(cfg, seed=TINY_MISTRAL_SEED, device='cpu')
        out['weights_sha256'] = np.array(weights_digest(sd))
        with tempfile.TemporaryDirectory() as tmp:
            tmp_path = Path(tmp)
            write_tiny_mistral_checkpoint(tmp_path / 'ckpt', window)
            encoder = AutoEncoder(AutoEncoderConfig(
                pretrained_model_name_or_path=str(tmp_path / 'ckpt'), quantization=False, eval_mode=True))
            assert type(encoder.model).__name__ == 'MistralModel'
            assert encoder.tokenizer.model_max_length == TINY_MISTRAL['max_position_embeddings']

            def loader() -> DataLoader:
                return DataLoader(InMemoryDataset(texts), batch_size=4, num_workers=0,
                                  collate_fn=DataCollator(encoder.tokenizer))

            for side in ('right', 'left'):
                encoder.tokenizer.padding_side = side
                key = f'{variant}/{side}'
                for i, batch in enumerate(loader()):
                    out[f'{key}/batch{i}/input_ids'] = batch['input_ids'].numpy()
                    out[f'{key}/batch{i}/attention_mask'] = batch['attention_mask'].numpy()
                    assert 'token_type_ids' not in batch
                    if i == 1 and key != 'window/left':   # batch 1 holds the truncated 320-token row
                        with torch.no_grad():
                            out[f'{key}/batch{i}/hidden'] = encoder.encode(batch).numpy()
                out['n_batches'] = np.array(i + 1)
                out[f'{key}/pooled/last_token'] = compute_embeddings(
                    loader(), encoder, LastTokenPooler(LastTokenPoolerConfig()))
                if side == 'right':
                    out[f'{key}/pooled/mean_normalized'] = compute_embeddings(
                        loader(), encoder, MeanPooler(MeanPoolerConfig()), normalize=True)
    np.savez_compressed(GOLDEN / 'mistral_tiny_golden.npz', **out)


TINY_MODERNBERT = dict(vocab_size=320, hidden_size=256, num_hidden_layers=4, num_attention_heads=4,
                       intermediate_size=384, max_position_embeddings=512, local_attention=32, norm_eps=1e-5,
                       pad_token_id=0, bos_token_id=1, eos_token_id=2, cls_token_id=1, sep_token_id=2,
                       initializer_range=0.05)
TINY_MODERNBERT_SEED = 1357


def tiny_modernbert_texts() -> list[str]:
    """12 texts behind modernbert_tiny_golden.npz: up to 300 words, so that the sliding window (|i - j| <= 16)
    and several 64-key chunks / two 128-row query tiles are exercised."""
    words = [f'w{i:03d}' for i in range(TINY_MODERNBERT['vocab_size'] - 4)]
    rng = np.random.default_rng(31)
    lengths = [5, 150, 33, 1, 64, 63, 300, 7, 127, 128, 200, 90]
    return [' '.join(rng.choice(words, size=n)) for n in lengths]


def write_tiny_modernbert_checkpoint(ckpt_dir: Path) -> None:
    from tokenizers import Tokenizer
    from tokenizers.models import WordLevel
    from tokenizers.pre_tokenizers import Whitespace
    from tokenizers.processors import TemplateProcessing
    from transformers import ModernBertConfig
    from transformers import ModernBertModel
    from transformers import PreTrainedTokenizerFast

    from distllm_b200.embed.encoders.weights import random_modernbert_state_dict

    words = [f'w{i:03d}' for i in range(TINY_MODERNBERT['vocab_size'] - 4)]
    vocab = {t: i for i, t in enumerate(['[PAD]', '[CLS]', '[SEP]', '[UNK]', *words])}
    cfg = ModernBertConfig(**TINY_MODERNBERT)
    sd = random_modernbert_state_dict(cfg, seed=TINY_MODERNBERT_SEED, device='cpu')
    model = ModernBertModel(cfg)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    raw = Tokenizer(WordLevel(vocab, unk_token='[UNK]'))
    raw.pre_tokenizer = Whitespace()
    raw.post_processor = TemplateProcessing(single='[CLS] $A [SEP]', special_tokens=[('[CLS]', 1), ('[SEP]', 2)])
    tok = PreTrainedTokenizerFast(tokenizer_object=raw, pad_token='[PAD]', cls_token='[CLS]', sep_token='[SEP]',
                                  unk_token='[UNK]', model_input_names=['input_ids', 'attention_mask'])
    model.eval().save_pretrained(ckpt_dir)
    tok.save_pretrained(ckpt_dir)


def make_modernbert_golden() -> None:
    """The reference's AutoEncoder (HF ModernBertModel: rotary per layer type, full / sliding-window attention,
    GeGLU) + MeanPooler / LastTokenPooler + compute_embeddings on a tiny seeded checkpoint (the family of
    examples/embed/workstation/modernbert_semchunk.yaml)."""
    from torch.utils.data import DataLoader
    from transformers import ModernBertConfig

    from distllm.embed.datasets.utils import DataCollator
    from distllm.embed.datasets.utils import InMemoryDataset
    from distllm.embed.embedders.full_sequence import compute_embeddings
    from distllm.embed.encoders.auto import AutoEncoder
    from distllm.embed.encoders.auto import AutoEncoderConfig
    from distllm.embed.poolers.last_token import LastTokenPooler
    from distllm.embed.poolers.last_token import LastTokenPoolerConfig
    from distllm.embed.poolers.mean import MeanPooler
    from distllm.embed.poolers.mean import MeanPoolerConfig
    from distllm_b200.embed.encoders.weights import random_modernbert_state_dict

    cfg = ModernBertConfig(**TINY_MODERNBERT)
    sd = random_modernbert_state_dict(cfg, seed=TINY_MODERNBERT_SEED, device='cpu')
    texts = tiny_modernbert_texts()
    out = {'n_texts': np.array(len(texts)), 'weights_sha256': np.array(weights_digest(sd))}
    with tempfile.TemporaryDirectory() as tmp:
        tmp_path = Path(tmp)
        write_tiny_modernbert_checkpoint(tmp_path / 'ckpt')
        encoder = AutoEncoder(AutoEncoderConfig(
            pretrained_model_name_or_path=str(tmp_path / 'ckpt'), quantization=False, eval_mode=True))
        assert type(encoder.model).__name__ == 'ModernBertModel'
        assert encoder.tokenizer.model_max_length == TINY_MODERNBERT['max_position_embeddings']

        def loader() -> DataLoader:
            return DataLoader(InMemoryDataset(texts), batch_size=4, num_workers=0,
                              collate_fn=DataCollator(encoder.tokenizer))

        for i, batch in enumerate(loader()):
            out[f'batch{i}/input_ids'] = batch['input_ids'].numpy()
            out[f'batch{i}/attention_mask'] = batch['attention_mask'].numpy()
            assert 'token_type_ids' not in batch
            if i == 1:    # holds the 300-word row
                with torch.no_grad():
                    out[f'batch{i}/hidden'] = encoder.encode(batch).numpy()
        out['n_batches'] = np.array(i + 1)
        out['pooled/mean_normalized'] = compute_embeddings(loader(), encoder, MeanPooler(MeanPoolerConfig()),
                                                           normalize=True)
        out['pooled/last_token'] = compute_embeddings(loader(), encoder, LastTokenPooler(LastTokenPoolerConfig()))
    np.savez_compressed(GOLDEN / 'modernbert_tiny_golden.npz', **out)


WORKER_DATASET = {'name': 'jsonl_chunk', 'buffer_size': 1, 'min_buffer_length': 20, 'batch_size': 5,
                  'num_data_workers': 0, 'pin_memory': False}
WORKER_EMBEDDER = {'name': 'semantic_chunk', 'breakpoint_percentile_threshold': 80, 'chunk_batch_size': 4,
                   'min_chunk_length': 10}


def worker_docs() -> list[dict]:
    """Three documents of 12-14 short sentences for the semantic-chunk worker golden."""
    words = tiny_bert_vocab()[5:]
    rng = np.random.default_rng(0)
    docs = []
    for d in range(3):
        sents = [('S' + ' '.join(rng.choice(words, size=rng.integers(5, 9))) + '. ') for _ in range(12 + d)]
        docs.append({'text': ''.join(sents), 'path': f'doc{d}'})
    return docs


def make_worker_golden() -> None:
    """The reference's own ``embedding_worker`` (distllm/distributed_embedding.py:23-80), file in -> files out,
    on the tiny BERT checkpoint: jsonl_chunk dataset -> semantic_chunk embedder -> mean pooler -> numpy writer.
    parsl / nltk are the stand-ins of oracle/ref_shims.py (the sentence splitter is the regex one on both
    sides)."""
    import json

    from oracle import ref_shims

    with tempfile.TemporaryDirectory() as tmp:
        tmp_path = Path(tmp)
        write_tiny_bert_checkpoint(tmp_path / 'ckpt')
        f = tmp_path / 'docs.jsonl'
        f.write_text('\n'.join(json.dumps(d) for d in worker_docs()))
        timers = ref_shims.run_embedding_worker(
            f, tmp_path / 'out',
            dataset_kwargs=dict(WORKER_DATASET),
            encoder_kwargs={'name': 'auto', 'pretrained_model_name_or_path': str(tmp_path / 'ckpt'),
                            'quantization': False, 'eval_mode': True},
            pooler_kwargs={'name': 'mean'},
            embedder_kwargs=dict(WORKER_EMBEDDER),
            writer_kwargs={'name': 'numpy'},
        )
        assert timers['computed-embeddings'] >= 0
        out = next((tmp_path / 'out').iterdir())
        emb = np.load(out / 'embeddings.npy')
        text = np.load(out / 'text.npy')
        meta = np.load(out / 'metadata.npy', allow_pickle=True)
        np.savez_compressed(GOLDEN / 'worker_golden.npz', embeddings=emb, text=text,
                            paths=np.array([m['path'] for m in meta]))


def main() -> None:
    sys.path.insert(0, str(REPO))
    from oracle import ref_shims

    print('reference:', ref_shims.install_reference())
    if ref_shims.reference_root() is None:
        raise SystemExit('golden vectors are made by the reference: no checkout found, set DISTLLM_REFERENCE')
    ref_shims.install()
    GOLDEN.mkdir(parents=True, exist_ok=True)
    torch.manual_seed(0)
    make_pool_golden()
    make_semantic_golden()
    make_bert_golden()
    make_esm_golden()
    make_mistral_golden()
    make_modernbert_golden()
    make_worker_golden()
    for f in sorted(GOLDEN.glob('*.npz')):
        print(f.name, f.stat().st_size, 'bytes')


if __name__ == '__main__':
    main()
