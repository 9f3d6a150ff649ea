"""Import the UNMODIFIED reference classes from a checkout of the reference project, with third-party stubs.

TEST INFRASTRUCTURE: the checkout is not part of this repository (it is looked for in
$VIDMEM_REFERENCE_ROOT, else in oracle/_ref/), so nothing that must run from the repository
alone (gpu tests, smoke(), bench.py) may import this module.  It is used by
oracle/gen_golden.py to produce tests/golden/ fixtures and by the CPU-only tests that
compare with the live reference when a checkout is present.

Missing third-party modules (langchain*, neo4j, sentence_transformers: SURVEY.md 8c) are
replaced with empty stand-ins in sys.modules; the reference's own code is executed as-is.
"""
from __future__ import annotations

import contextlib
import os
import sys
import tempfile
import types

REFERENCE_ROOT = os.environ.get("VIDMEM_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "components"))


class _Anything:
    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        return _Anything()


def _stub(name: str, **attrs) -> None:
    if name in sys.modules:
        return
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    def _missing(attr):
        # any ordinary symbol resolves to a dummy class; dunders (__file__, __path__, ...) must stay absent so
        # that tools which introspect sys.modules (hypothesis, importlib) see a normal, file-less module
        if attr.startswith("__") and attr.endswith("__"):
            raise AttributeError(attr)
        return _Anything

    m.__getattr__ = _missing
    sys.modules[name] = m
    if "." in name:
        parent, child = name.rsplit(".", 1)
        _stub(parent)
        setattr(sys.modules[parent], child, m)


@contextlib.contextmanager
def _cwd_tmp():
    # src/core/logger.py:42-43 creates ./logs at import; keep that out of the repo
    old = os.getcwd()
    d = tempfile.mkdtemp(prefix="vidmem_ref_")
    os.chdir(d)
    try:
        yield d
    finally:
        os.chdir(old)


_loaded = {}


def load():
    """Returns a dict with the reference's PreLLMInjector, HybridRetriever, EmbeddingUtils and
    prune.Graph classes (unmodified)."""
    if _loaded:
        return _loaded
    if not available():
        raise RuntimeError("reference checkout not present at " + REFERENCE_ROOT)
    for name in ("langchain_core", "langchain_core.prompts", "langchain_core.language_models",
                 "langchain_core.documents", "langchain_core.messages", "langchain_core.output_parsers",
                 "langchain_text_splitters", "langchain_experimental",
                 "langchain_experimental.graph_transformers", "langchain_openai", "neo4j", "neo4j.exceptions",
                 "sentence_transformers", "json_repair", "nltk", "rapidfuzz"):
        try:
            __import__(name)
        except Exception:
            _stub(name)
    os.environ.setdefault("VIDGRAPH_LOG_LEVEL", "ERROR")
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        with _cwd_tmp():
            from src.components.pre_llm_injector import PreLLMInjector
            from src.pipeline.retriever_hybrid import HybridRetriever
            from src.utils.embedding_utils import EmbeddingUtils
            from src.pipeline import prune as prune_mod
            from src.core.config import EmbedderConfig
    finally:
        sys.path.remove(REFERENCE_ROOT)
    _loaded.update(PreLLMInjector=PreLLMInjector, HybridRetriever=HybridRetriever, EmbeddingUtils=EmbeddingUtils,
                   Graph=prune_mod.Graph, EmbedderConfig=EmbedderConfig)
    return _loaded


def make_injector(top_k: int, top_k2: int = 2):
    """A PreLLMInjector instance without running its constructor (which needs an LLM)."""
    ref = load()
    inj = object.__new__(ref["PreLLMInjector"])
    inj.embedder_config = types.SimpleNamespace(top_k_chunk_with_batch_similarity=top_k, top_k_similar_batch=top_k2)
    return inj


def run_batch_similarities(queries, store_dict, top_k: int):
    """Runs the reference's own _calculate_batch_similarities (pre_llm_injector.py:346-372) with
    _get_chunk_embeddings replaced by a coroutine returning `store_dict`."""
    import asyncio

    inj = make_injector(top_k)

    async def fake_get(_handler):
        return store_dict

    inj._get_chunk_embeddings = fake_get
    return asyncio.run(inj._calculate_batch_similarities(queries, object()))


def make_graph(encode):
    """prune.Graph without its constructor (which downloads a SentenceTransformer)."""
    ref = load()
    g = object.__new__(ref["Graph"])
    g.embedding_model = types.SimpleNamespace(encode=encode)
    return g
