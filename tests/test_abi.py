"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol include/digat_sm100.h
declares; the Python module mirrors the reference's parameter names; no compute calls (no GPU here)."""
import ctypes
import os
import re

import pytest
import torch

from tests.helpers import CASES, ROOT, case_inputs, check_hashes, load_golden


def _declared_symbols():
    src = open(os.path.join(ROOT, 'include', 'digat_sm100.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(digat_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol_at_abi_7():
    from digat_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared_symbols()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), 'libdigat_sm100.so does not export ' + n
    bound = set(_lib.SIGNATURES) | {'digat_last_error'}
    assert set(names) == bound, 'ctypes SIGNATURES out of sync with the header: %s' % (set(names) ^ bound)
    assert _lib.load().digat_abi_version() == 7


def test_no_gpu_fails_loudly():
    from digat_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(RuntimeError):
        _lib.require_device(0)
    assert _lib.load().digat_device_check(None) < 0
    assert 'CUDA' in _lib.last_error() or 'device' in _lib.last_error()


def test_invalid_arguments_return_error_codes():
    """Argument validation happens before any CUDA call, so it can be exercised without a GPU."""
    from digat_b200 import _lib
    lib = _lib.load()
    assert lib.digat_linear_f32(None, 4, None, 4, None, None, 4, 1, 1, 4, 0, None, 1, 0, 0, 0, None) == -1
    assert 'null' in _lib.last_error()
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    p = (p + 15) & ~15
    assert lib.digat_linear_f32(p, 6, p, 8, None, p, 8, 1, 1, 6, 0, None, 1, 0, 0, 0, None) == -1        # K not multiple of 4
    assert lib.digat_graph_layer_fwd(p, 12, p, p, p, p, 1, 500, 4, None, 1.0, None, None, None, None, 0, None, None, 0, None, None, None, None, None, None, None) == -1   # n too large
    assert lib.digat_attention_pool_fwd(p, 8, 8, None, p, 8, p, None, p, 8, None, None, 1, 1000, 8, None) == -1


def test_state_dict_names_match_reference_layout():
    from digat_b200 import synth
    from digat_b200.graphEncoders import DIGAT
    cfg = synth.make_config(graph_depth=2)
    m = DIGAT(cfg, 400)
    sd = synth.make_state_dict(cfg)
    assert set(m.state_dict().keys()) == set(sd.keys())
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    m.load_state_dict(sd)
    m.initialize()
    assert float(m.topic_node_embedding.abs().sum()) == 0.0
    assert m.max_history_num == 50 and m.category_num == 19 and m.user_graph_size == 68


def test_state_dict_names_match_imported_reference():
    """The reference's DIGAT loaded the seeded weights of every golden case with a strict ``load_state_dict`` (every
    name, every shape) when the vectors were generated (oracle/make_golden.py), and each fixture records a hash of every
    weight under its name: those names are the reference's state-dict layout, and the hashes pin the weights loaded."""
    from digat_b200.graphEncoders import DIGAT
    for name in CASES:
        cfg, sd, _, batch = case_inputs(name)
        _, meta = load_golden(name)
        check_hashes(meta, sd, batch)
        ref_names = {k[len('w:'):] for k in meta if k.startswith('w:')}
        ours = DIGAT(cfg, 400)
        os_ = ours.state_dict()
        assert set(os_.keys()) == ref_names, name
        for k in os_:
            assert tuple(os_[k].shape) == tuple(sd[k].shape), (name, k)
        ours.load_state_dict(sd)


def _header_param_count(name):
    src = open(os.path.join(ROOT, 'include', 'digat_sm100.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    m = re.search(r'\b%s\s*\(([^)]*)\)\s*;' % re.escape(name), src)
    assert m, name + ' is not declared in the header'
    params = m.group(1).strip()
    return 0 if params in ('', 'void') else len(params.split(','))


def test_ctypes_signatures_have_the_arity_of_the_header():
    from digat_b200 import _lib
    for name, argtypes in _lib.SIGNATURES.items():
        assert len(argtypes) == _header_param_count(name), name


def test_documented_ctypes_stub_matches_header():
    """INTEGRATION.md shows the binding a maintainer would write for digat_graph_layer_fwd: its argtypes list and its
    example call must have exactly the parameters the header declares (a stale stub is undefined behaviour)."""
    doc = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    block = re.search(r'lib\.digat_graph_layer_fwd\.argtypes = \[(.*?)\]', doc, flags=re.S).group(1)
    block = re.sub(r'#[^\n]*', '', block)
    n_types = len([t for t in block.replace('\n', ' ').split(',') if t.strip()])
    call = re.search(r'rc = lib\.digat_graph_layer_fwd\((.*?)\)\nif rc', doc, flags=re.S).group(1)
    depth, n_args = 0, 1
    for ch in call:
        depth += ch in '([' 
        depth -= ch in ')]'
        n_args += ch == ',' and depth == 0
    want = _header_param_count('digat_graph_layer_fwd')
    assert n_types == want and n_args == want, (n_types, n_args, want)
