"""Import the UNMODIFIED reference classes from a checkout of the upstream project: oracle/_ref (git-ignored), or the
directory SCONE_REFERENCE_ROOT names.

TEST INFRASTRUCTURE ONLY.  The reference is not part of this repository, so
nothing in ``-m gpu`` tests, ``smoke()`` or ``bench.py`` may call this; it is
used by ``tests/golden/make_golden.py`` (fixture generation) and by the CPU
test that runs the reference side by side with the oracle when a checkout is present.

The reference does not import cleanly as shipped: ``scone/utils/__init__.py:3``
imports a module that does not exist (``scone.utils.cloud``), which breaks
``scone.inference`` via ``scone/inference/engine.py:11``.  We never edit the
reference; we load the two hot-path files directly by path, under private
module names, so none of the broken package ``__init__`` files run.
"""

from __future__ import annotations

import importlib.util
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("SCONE_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "scone", "tokenization", "n_gram_extractor.py"))


def _load(name: str, relpath: str):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    """Returns (NGramExtractor, EmbeddingCache) classes of the reference."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REFERENCE_ROOT}: put the upstream scone repository there or "
                           "name it in SCONE_REFERENCE_ROOT")
    # embedding_cache.py does `from scone.tokenization.n_gram_extractor import NGramExtractor`.
    # Provide bare package shells (no __init__ executed) so that import resolves
    # to the file we load by path.
    for pkg in ("scone", "scone.tokenization", "scone.inference"):
        if pkg not in sys.modules:
            shell = types.ModuleType(pkg)
            shell.__path__ = []  # mark as package, but with nothing discoverable
            sys.modules[pkg] = shell
    nge = _load("scone.tokenization.n_gram_extractor", "scone/tokenization/n_gram_extractor.py")
    ec = _load("scone.inference.embedding_cache", "scone/inference/embedding_cache.py")
    return nge.NGramExtractor, ec.EmbeddingCache
