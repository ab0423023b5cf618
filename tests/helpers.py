"""Shared helpers for the parity tests: rebuild the seeded golden-case inputs and check their hashes."""
import hashlib
import json
import os

import numpy as np

from digat_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

# must match oracle/make_golden.py::CASES
CASES = {
    'default_n3_L3': (3, 2, 3, 6, True, 0.3),
    'code_default_n5_L2': (5, 2, 2, 4, False, 0.3),
    'wide_n8_L7': (8, 2, 7, 2, False, 0.3),
    'unit_normal_n3_L3': (3, 2, 3, 4, False, 1.0),
}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def case_inputs(name):
    """Same construction as oracle/make_golden.py::case_inputs (kept separate: tests must not need the reference code)."""
    N, hops, L, rows, keep, scale = CASES[name]
    cfg = synth.make_config(SAG_neighbors=N, SAG_hops=hops, graph_depth=L)
    sd = synth.make_state_dict(cfg, seed=11)
    corpus = synth.make_corpus(cfg, n_news=300, n_behaviors=12, mean_candidates=3.0, seed=5, emb_scale=scale)
    rng = np.random.Generator(np.random.PCG64(99))
    ids = rng.choice(corpus.pair_behavior.shape[0], size=rows, replace=False)
    empty = np.nonzero(~corpus.user_category_mask.any(axis=1))[0]
    if len(empty):
        hit = np.nonzero(corpus.pair_behavior == empty[0])[0]
        if len(hit):
            ids[0] = hit[0]
    batch = synth.make_batch(corpus, np.sort(ids))
    return cfg, sd, corpus, batch


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, 'encoder_%s.npz' % name))
    meta = json.loads(bytes(z['meta']).decode())
    return z, meta


def check_hashes(meta, sd, batch):
    for k, v in sd.items():
        assert meta['w:' + k] == sha(v.numpy()), 'synthetic weight %s drifted from the golden fixture' % k
    for k, v in batch.items():
        assert meta['x:' + k] == sha(v.numpy()), 'synthetic input %s drifted from the golden fixture' % k


def rel_err(a, b):
    """max |a-b| / max|b| -- relative to the tensor's scale (logits can be individually near zero)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def ulp_distance(a, b):
    """Distance between two fp32 arrays in units in the last place (ordered-integer view of the IEEE bit patterns)."""
    def key(x):
        u = np.ascontiguousarray(np.asarray(x, dtype=np.float32)).view(np.int32).astype(np.int64)
        return np.where(u < 0, -(u & 0x7FFFFFFF), u)
    return np.abs(key(a) - key(b))


def err_stats(got, ref, terms=None, floor_frac=1e-3):
    """Error of ``got`` against ``ref`` reported three ways (tests gate on 'max_norm'; the others are printed and, where a
    test says so, gated too):
      max_norm : max|got-ref| / max|ref|                                  (the scale of the tensor)
      per_elem : max over elements of |got-ref| / max(|ref|, floor),  floor = floor_frac * max|ref|   (per-logit error;
                 the floor is stated because a single logit may be arbitrarily close to zero)
      cond     : max over elements of |got-ref| / terms,  terms[i] = sum_d |x_d * y_d| of the dot product that forms
                 element i (the magnitude fp32 rounding acts on: |logit| <= terms); only when ``terms`` is given
      max_ulp  : largest distance in fp32 units in the last place."""
    g = np.asarray(got, dtype=np.float64)
    r = np.asarray(ref, dtype=np.float64)
    scale = max(float(np.max(np.abs(r))), 1e-30)
    d = np.abs(g - r)
    out = {'max_norm': float(d.max() / scale),
           'per_elem': float(np.max(d / np.maximum(np.abs(r), floor_frac * scale))),
           'floor': floor_frac * scale,
           'max_ulp': int(ulp_distance(got, ref).max())}
    if terms is not None:
        out['cond'] = float(np.max(d / np.maximum(np.asarray(terms, dtype=np.float64), 1e-30)))
    return out


def fmt_stats(s):
    return ', '.join('%s %s' % (k, ('%d' % v) if k == 'max_ulp' else ('%.2e' % v)) for k, v in s.items())


# must match oracle/make_golden.py::ABLATION_CASES
ABLATION_KINDS = ('wo_SA', 'Seq_SA', 'wo_interaction', 'news_graph_wo_inter', 'user_graph_wo_inter')
ABLATION_CASES = {'n3_L2': (3, 2, 2, 5), 'n5_L3': (5, 2, 3, 3)}


def ablation_inputs(kind, case):
    """Same construction as oracle/make_golden.py::ablation_inputs."""
    N, hops, L, rows = ABLATION_CASES[case]
    cfg = synth.make_config(SAG_neighbors=N, SAG_hops=hops, graph_depth=L, graph_encoder=kind)
    sd = synth.make_ablation_state_dict(kind, cfg, seed=13)
    corpus = synth.make_corpus(cfg, n_news=300, n_behaviors=12, mean_candidates=3.0, seed=6)
    rng = np.random.Generator(np.random.PCG64(98))
    ids = rng.choice(corpus.pair_behavior.shape[0], size=rows, replace=False)
    empty = np.nonzero(~corpus.user_category_mask.any(axis=1))[0]
    if len(empty):
        hit = np.nonzero(corpus.pair_behavior == empty[0])[0]
        if len(hit):
            ids[0] = hit[0]
    return cfg, sd, synth.make_batch(corpus, np.sort(ids))


def load_ablation_golden(kind, case):
    z = np.load(os.path.join(GOLDEN, 'ablation_%s_%s.npz' % (kind, case)))
    return z, json.loads(bytes(z['meta']).decode())


def msa_inputs():
    """Same construction as oracle/make_golden.py::msa_inputs."""
    cfg = synth.make_text_config()
    sd = synth.make_msa_state_dict(cfg, seed=5)
    tok, mask = synth.make_titles(cfg, 24, seed=2)
    return cfg, sd, tok.view(4, 6, -1), mask.view(4, 6, -1)


def cnn_inputs(method):
    """Same construction as oracle/make_golden.py::cnn_inputs."""
    cfg = synth.make_text_config(cnn_method=method, cnn_kernel_num=384 if method == 'group3' else 400)
    sd = synth.make_cnn_state_dict(cfg, seed=6)
    tok, mask = synth.make_titles(cfg, 24, seed=3)
    return cfg, sd, tok.view(4, 6, -1), mask.view(4, 6, -1)
