"""TEST INFRASTRUCTURE ONLY -- import the UNMODIFIED reference modules from a checkout of the original DIGAT code, which
is not part of this repository: set ``DIGAT_REFERENCE_ROOT`` to its directory.

This loader is used only by ``oracle/make_golden.py`` (fixture generation) and by the CPU tests of
``tests/test_reference_dropin.py``, which skip when no reference checkout is given.

Three modules the reference imports are not installed and there is no network (SURVEY.md section 8c):
``torchtext`` (MIND_corpus.py:8), ``sentence_transformers`` (construct_SAG.py:4) -- both off the hot path, stubbed
with empty modules -- and ``torch_scatter`` (graphEncoders.py:7), replaced by ``oracle/scatter_shim.py``.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get('DIGAT_REFERENCE_ROOT', '')


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, 'graphEncoders.py'))


def load_reference():
    """Returns the reference's (graphEncoders, layers, model, evaluate) modules."""
    if not reference_available():
        raise RuntimeError('reference tree not found: set DIGAT_REFERENCE_ROOT to a checkout of the original DIGAT code')
    from . import scatter_shim
    if 'torchtext' not in sys.modules:
        tt = types.ModuleType('torchtext')
        ttv = types.ModuleType('torchtext.vocab')
        ttv.GloVe = object
        tt.vocab = ttv
        sys.modules['torchtext'] = tt
        sys.modules['torchtext.vocab'] = ttv
    if 'sentence_transformers' not in sys.modules:
        st = types.ModuleType('sentence_transformers')
        st.SentenceTransformer = object
        sys.modules['sentence_transformers'] = st
    if 'torch_scatter' not in sys.modules:
        ts = types.ModuleType('torch_scatter')
        ts.scatter_sum = scatter_shim.scatter_sum
        ts.scatter_softmax = scatter_shim.scatter_softmax
        sys.modules['torch_scatter'] = ts
    if REFERENCE_ROOT not in sys.path:
        sys.path.append(REFERENCE_ROOT)
    import importlib
    # the reference modules import each other by bare name (``from layers import ...``), so they are imported
    # through the normal machinery with the reference root appended (not prepended) to sys.path
    mods = {name: importlib.import_module(name) for name in ('layers', 'graphEncoders', 'evaluate', 'construct_SAG')}
    return mods['graphEncoders'], mods['layers'], mods['evaluate'], mods['construct_SAG']
