"""Run the UNMODIFIED reference (ramanathanlab/distllm) on CPU.  TEST / BENCH INFRASTRUCTURE ONLY.

The reference is pure Python.  ``install_reference`` copies its ``distllm`` package from an unmodified
checkout (``$DISTLLM_REFERENCE``, by default ``/root/reference``) into the git-ignored ``oracle/_ref``
(``__graft_entry__.build()`` does so wherever that checkout exists); everything here imports it from there.

Two of its import-time dependencies are absent from this image and are replaced by the smallest
stand-ins that let ``distllm.distributed_embedding.embedding_worker`` run (SURVEY 8c):

  * ``parsl``  imported at module scope by distllm/distributed_embedding.py:10 and distllm/parsl.py:16-23;
               never used on the worker path -> empty classes
  * ``nltk``   distllm/embed/datasets/jsonl_chunk.py:26-28 needs
               ``nltk.tokenize.PunktSentenceTokenizer().span_tokenize``; Punkt's model cannot be installed
               offline -> a regex span tokenizer (sentence end = ``.!?`` + whitespace + capital/digit).  The
               synthetic texts used with it end every sentence with ". " followed by a capital, which any
               splitter cuts identically.

Nothing here touches distllm_b200: the reference arm runs none of this repository's models or kernels.
"""

from __future__ import annotations

import contextlib
import io
import os
import re
import shutil
import sys
import tempfile
import types
from pathlib import Path

REPO = Path(__file__).resolve().parents[1]
REF_ROOT = REPO / 'oracle' / '_ref'
DEFAULT_SOURCE = Path('/root/reference')   # where the unmodified checkout is looked for without $DISTLLM_REFERENCE

_BOUNDARY = re.compile(r'[.!?]["\')\]]*\s+(?=[A-Z0-9"\'(\[])')


def reference_root() -> Path | None:
    """Directory to put on ``sys.path`` so that ``import distllm`` finds the unmodified reference."""
    if (REF_ROOT / 'distllm' / 'distributed_embedding.py').exists():
        return REF_ROOT
    return None


def install_reference() -> str:
    """Copy the reference's ``distllm`` package from ``$DISTLLM_REFERENCE`` (default ``DEFAULT_SOURCE``) into
    ``oracle/_ref`` (what ``bench.py --impl reference`` and its ``cpu_baseline`` leg run; without it they time
    the oracle port).
    A plain copy is the whole install: the package is pure Python, and its dependency pins (parsl, nltk,
    bitsandbytes, faiss-gpu ...) are not needed on the embedding path, where the stand-ins below replace
    the two it imports.  File modes are not copied, so a read-only source gives a removable copy."""
    if reference_root() is not None:
        return f'present: {REF_ROOT}'
    src = os.environ.get('DISTLLM_REFERENCE')
    pkg = Path(src or DEFAULT_SOURCE) / 'distllm'
    if not (pkg / 'distributed_embedding.py').exists():
        if src:
            raise RuntimeError(f'$DISTLLM_REFERENCE={src} is not a distllm checkout')
        return f'not installed (no checkout at {DEFAULT_SOURCE}); the CPU arm runs the oracle port'
    tmp = Path(tempfile.mkdtemp(prefix='_ref.', dir=REF_ROOT.parent))
    try:
        shutil.copytree(pkg, tmp / 'distllm', copy_function=shutil.copyfile,
                        ignore=shutil.ignore_patterns('__pycache__'))
        for d, _, _ in os.walk(tmp):
            os.chmod(d, 0o755)
        shutil.rmtree(REF_ROOT, ignore_errors=True)   # an incomplete earlier copy
        os.replace(tmp, REF_ROOT)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)        # gone already unless the copy failed
    return f'installed: {REF_ROOT}'


def _regex_spans(text: str) -> list[tuple[int, int]]:
    spans = []
    start = 0
    for m in _BOUNDARY.finditer(text):
        stop = m.start() + len(m.group().rstrip())
        spans.append((start, stop))
        start = m.end()
    if start < len(text):
        spans.append((start, len(text.rstrip()) if text.rstrip() else len(text)))
    return [(s, e) for s, e in spans if e > s]


def _stub_parsl() -> None:
    if 'parsl' in sys.modules:
        return
    try:
        import parsl  # noqa: F401

        return
    except ImportError:
        pass
    layout = {
        'parsl': [],
        'parsl.concurrent': ['ParslPoolExecutor'],
        'parsl.addresses': ['address_by_hostname'],
        'parsl.config': ['Config'],
        'parsl.executors': ['HighThroughputExecutor'],
        'parsl.launchers': ['MpiExecLauncher', 'SrunLauncher'],
        'parsl.providers': ['LocalProvider', 'PBSProProvider', 'SlurmProvider'],
    }
    for name, members in layout.items():
        mod = types.ModuleType(name)
        mod.__path__ = []  # type: ignore[attr-defined]
        for member in members:
            setattr(mod, member, type(member, (), {}))
        sys.modules[name] = mod
    for name in layout:
        if '.' in name:
            setattr(sys.modules['parsl'], name.split('.')[1], sys.modules[name])


def _stub_nltk() -> None:
    if 'nltk' in sys.modules:
        return
    try:
        import nltk  # noqa: F401

        return
    except ImportError:
        pass

    class PunktSentenceTokenizer:  # noqa: D401  minimal stand-in, see module docstring
        def span_tokenize(self, text: str):
            return iter(_regex_spans(text))

    nltk = types.ModuleType('nltk')
    tokenize = types.ModuleType('nltk.tokenize')
    tokenize.PunktSentenceTokenizer = PunktSentenceTokenizer  # type: ignore[attr-defined]
    nltk.tokenize = tokenize  # type: ignore[attr-defined]
    nltk.__path__ = []  # type: ignore[attr-defined]
    sys.modules['nltk'] = nltk
    sys.modules['nltk.tokenize'] = tokenize


def install(root: Path | None = None) -> Path:
    """Make ``import distllm`` resolve to the unmodified reference; returns the root used."""
    root = root or reference_root()
    if root is None:
        raise RuntimeError('the reference is not installed in oracle/_ref (see install_reference)')
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    _stub_parsl()
    _stub_nltk()
    return root


_TIMER_LINE = re.compile(r'\[timer\] \[([^\]]+)\] in \[([0-9.]+)\] seconds')


def run_embedding_worker(input_path: Path, output_dir: Path, **kwargs) -> dict[str, float]:
    """Call the reference's ``embedding_worker`` (distllm/distributed_embedding.py:23-80) and return its
    own ``[timer]`` readings (distllm/timer.py:156-162) keyed by the first tag, e.g.
    ``{'loaded-encoder': 0.51, 'computed-embeddings': 12.3, ...}``."""
    install()
    from distllm.distributed_embedding import embedding_worker

    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        embedding_worker(input_path=Path(input_path), output_dir=Path(output_dir), **kwargs)
    timers: dict[str, float] = {}
    for tags, seconds in _TIMER_LINE.findall(buf.getvalue()):
        timers[tags.split()[0]] = float(seconds)
    if 'computed-embeddings' not in timers:
        raise RuntimeError(f'no [timer] [computed-embeddings ...] line in the reference output:\n{buf.getvalue()}')
    return timers
