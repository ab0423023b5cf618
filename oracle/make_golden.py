"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the UNMODIFIED reference code (not in this repository).

Run:  DIGAT_REFERENCE_ROOT=<checkout of the original DIGAT code> python -m oracle.make_golden     (writes tests/golden/)

Inputs are NOT stored: they are rebuilt from seeds by ``digat_b200.synth`` (numpy PCG64).  Each fixture stores a
sha256 of every input/weight array so that a drift of the generator is detected instead of silently comparing
different problems.  Outputs stored per case:

* ``ref32_*``  -- the reference modules run in fp32 on CPU (the parity target);
* ``ref64_*``  -- the same modules after ``.double()`` (ground truth for error budgeting);
* integer cases -- construct_SAG.generate_news_graph on a seeded similarity table; evaluate.scoring metrics.
"""
import hashlib
import io
import json
import os
import sys
import zipfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from digat_b200 import synth  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')

# name -> (SAG_neighbors, SAG_hops, depth, rows, keep_intermediates, emb_scale)
CASES = {
    'default_n3_L3': (3, 2, 3, 6, True, 0.3),
    'code_default_n5_L2': (5, 2, 2, 4, False, 0.3),
    'wide_n8_L7': (8, 2, 7, 2, False, 0.3),
    'unit_normal_n3_L3': (3, 2, 3, 4, False, 1.0),
}


def sha(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(a.tobytes()).hexdigest()


def case_inputs(name):
    N, hops, L, rows, keep, scale = CASES[name]
    cfg = synth.make_config(SAG_neighbors=N, SAG_hops=hops, graph_depth=L)
    sd = synth.make_state_dict(cfg, seed=11)
    corpus = synth.make_corpus(cfg, n_news=300, n_behaviors=12, mean_candidates=3.0, seed=5, emb_scale=scale)
    # rows chosen to include an empty-history behaviour and an isolated news if present
    rng = np.random.Generator(np.random.PCG64(99))
    ids = rng.choice(corpus.pair_behavior.shape[0], size=rows, replace=False)
    empty = np.nonzero(~corpus.user_category_mask.any(axis=1))[0]
    if len(empty):
        hit = np.nonzero(corpus.pair_behavior == empty[0])[0]
        if len(hit):
            ids[0] = hit[0]
    batch = synth.make_batch(corpus, np.sort(ids))
    return cfg, sd, corpus, batch


def save_golden(path, **arrays):
    """``np.savez`` with LZMA-compressed members, which ``np.load`` reads like any .npz: float vectors pack about 30%
    smaller than with ``np.savez_compressed``, which keeps every fixture under 1 MB."""
    with zipfile.ZipFile(path, 'w', compression=zipfile.ZIP_LZMA) as zf:
        for k, v in arrays.items():
            with zf.open(k + '.npy', 'w', force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(v), allow_pickle=False)


def input_hashes(sd, batch):
    h = {('w:' + k): sha(v.numpy()) for k, v in sd.items()}
    h.update({('x:' + k): sha(v.numpy()) for k, v in batch.items()})
    return h


def run_reference(ge, cfg, sd, batch, dtype, keep):
    m = ge.DIGAT(cfg, 400)
    m.load_state_dict(sd)
    m = m.to(dtype).eval()
    f = lambda t: t.to(dtype) if t.is_floating_point() else t
    b = {k: f(v) for k, v in batch.items()}
    out = {}
    with torch.no_grad():
        c_n0 = m.compute_news_graph_context(b['news_graph_embeddings'], b['news_graph_mask'])
        args = (b['news_graph_embeddings'], b['news_graph'], b['news_graph_mask'], b['user_news_embedding'],
                b['user_graph'], b['user_category_mask'], b['user_category_indices'])
        cn, cu = m.inference(*args, c_n0)
        fn, fu = m.forward(*args)
        out['c_n0'] = c_n0
        out['news_ctx'], out['user_ctx'] = cn, cu
        out['fwd_news_ctx'], out['fwd_user_ctx'] = fn, fu
        out['logits'] = (cu * cn).sum(dim=1)
        if keep:
            X_u = torch.cat([b['user_news_embedding'], m.topic_node_embedding.unsqueeze(0).expand(cn.shape[0], -1, -1)], 1)
            c_u0 = m.compute_user_graph_context(X_u, b['user_category_mask'], b['user_category_indices'], c_n0)
            out['c_u0'] = c_u0
            out['Y_news_l0'] = m.compute_news_graph_embeddings(0, b['news_graph_embeddings'], b['news_graph'], c_u0)
            out['Y_user_l0'] = m.compute_user_graph_embeddings(0, X_u, b['user_graph'], c_n0)
    return {k: v.numpy() for k, v in out.items()}


def make_encoder_cases(ge):
    for name, (N, hops, L, rows, keep, scale) in CASES.items():
        cfg, sd, corpus, batch = case_inputs(name)
        payload = {'meta': np.frombuffer(json.dumps(input_hashes(sd, batch)).encode(), dtype=np.uint8)}
        for tag, dt in (('ref32_', torch.float32), ('ref64_', torch.float64)):
            for k, v in run_reference(ge, cfg, sd, batch, dt, keep).items():
                payload[tag + k] = v
        save_golden(os.path.join(GOLDEN, 'encoder_%s.npz' % name), **payload)
        print(name, {k: v.shape for k, v in payload.items() if k != 'meta'})


ABLATION_CLASSES = {'wo_SA': 'wo_SA', 'Seq_SA': 'Seq_SA', 'wo_interaction': 'wo_interaction',
                    'news_graph_wo_inter': 'News_graph_wo_inter', 'user_graph_wo_inter': 'User_graph_wo_inter'}
# name -> (SAG_neighbors, SAG_hops, depth, rows)
ABLATION_CASES = {'n3_L2': (3, 2, 2, 5), 'n5_L3': (5, 2, 3, 3)}


def ablation_inputs(kind, case):
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


def make_ablation_cases(ge):
    """The five ablation encoders of the unmodified reference (graphEncoders.py:201-842): inference, forward (eval) and
    the first user/news layer outputs."""
    for kind, cls in ABLATION_CLASSES.items():
        for case in ABLATION_CASES:
            cfg, sd, batch = ablation_inputs(kind, case)
            payload = {'meta': np.frombuffer(json.dumps(input_hashes(sd, batch)).encode(), dtype=np.uint8)}
            for tag, dt in (('ref32_', torch.float32), ('ref64_', torch.float64)):
                m = getattr(ge, cls)(cfg, 400)
                m.load_state_dict(sd)
                m = m.to(dt).eval()
                b = {k: (v.to(dt) if v.is_floating_point() else v) for k, v in batch.items()}
                args = (b['news_graph_embeddings'], b['news_graph'], b['news_graph_mask'], b['user_news_embedding'],
                        b['user_graph'], b['user_category_mask'], b['user_category_indices'])
                with torch.no_grad():
                    if kind == 'wo_SA':
                        c_n0 = torch.zeros(args[0].shape[0], 400, dtype=dt)
                    elif kind == 'Seq_SA':
                        c_n0 = m.compute_news_sequence_context(args[0], args[2])
                    else:
                        c_n0 = m.compute_news_graph_context(args[0], args[2])
                    cn, cu = m.inference(*args, c_n0)
                    fn, fu = m.forward(*args)
                    out = {'c_n0': c_n0, 'news_ctx': cn, 'user_ctx': cu, 'fwd_news_ctx': fn, 'fwd_user_ctx': fu,
                           'logits': (cu * cn).sum(dim=1)}
                for k, v in out.items():
                    payload[tag + k] = v.numpy()
            save_golden(os.path.join(GOLDEN, 'ablation_%s_%s.npz' % (kind, case)), **payload)
            print(kind, case, {k: v.shape for k, v in payload.items() if k != 'meta'})


def msa_inputs():
    cfg = synth.make_text_config()
    sd = synth.make_msa_state_dict(cfg, seed=5)
    tok, mask = synth.make_titles(cfg, 24, seed=2)
    return cfg, sd, tok.view(4, 6, -1), mask.view(4, 6, -1)


def make_msa_case():
    """newsEncoders.MSA of the unmodified reference (eval mode).  Its constructor reads the preprocessed word-embedding pickle
    from the working directory (newsEncoders.py:14-15): a temporary one is provided, then the seeded weights are loaded."""
    import importlib
    import pickle
    import tempfile
    cfg, sd, tok, mask = msa_inputs()
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            with open('word_embedding-%s-%s-%s-%s.pkl' % (cfg.word_threshold, cfg.word_embedding_dim, cfg.max_title_length,
                                                           cfg.dataset), 'wb') as f:
                pickle.dump(torch.zeros(cfg.vocabulary_size, cfg.word_embedding_dim), f)
            ne = importlib.import_module('newsEncoders')
            payload = {'meta': np.frombuffer(json.dumps({('w:' + k): sha(v.numpy()) for k, v in sd.items()} |
                                                        {'x:title_text': sha(tok.numpy()), 'x:title_mask': sha(mask.numpy())}).encode(),
                                             dtype=np.uint8)}
            for tag, dt in (('ref32_', torch.float32), ('ref64_', torch.float64)):
                m = ne.MSA(cfg)
                m.load_state_dict(sd)
                m = m.to(dt).eval()
                with torch.no_grad():
                    payload[tag + 'news'] = m(tok, mask.to(dt)).numpy()
        finally:
            os.chdir(cwd)
    save_golden(os.path.join(GOLDEN, 'news_encoder_msa.npz'), **payload)
    print('news_encoder_msa', payload['ref32_news'].shape)


def make_sag_case(sag):
    """construct_SAG.generate_news_graph on a seeded similarity table (integer golden vectors)."""
    rng = np.random.Generator(np.random.PCG64(7))
    n_news, top_M, hop = 60, 4, 2
    n_nodes = synth.sag_size(top_M, hop)
    ids = {'<PAD>': 0}
    for k in range(1, n_news):
        ids['N%d' % k] = k
    sim_tbl = np.zeros((n_news, top_M, 2), dtype=np.float64)
    sim_dict = {}
    for k in range(1, n_news):
        m = int(rng.integers(0, top_M + 1))
        others = rng.choice(np.arange(1, n_news), size=m, replace=False)
        cos = np.sort(rng.uniform(0.3, 1.0, size=m))[::-1]
        sim_dict['N%d' % k] = [['N%d' % o, float(c)] for o, c in zip(others, cos)]
        sim_tbl[k, :m, 0] = others
        sim_tbl[k, :m, 1] = cos
        sim_tbl[k, m:, 0] = -1
    node, graph, mask = sag.generate_news_graph('synthetic', sim_dict, ids, top_M, hop, n_nodes)
    save_golden(os.path.join(GOLDEN, 'sag_bfs.npz'), sim=sim_tbl, top_M=top_M, hop=hop, n_nodes=n_nodes,
                threshold=sag.similarity_threshold, node=node, graph=graph, mask=mask)
    print('sag_bfs', node.shape, int(mask.sum()))


def make_metric_case(ev):
    """evaluate.scoring on seeded scores (rank files written exactly as util.py:70-80 does)."""
    rng = np.random.Generator(np.random.PCG64(3))
    n_imp = 40
    sizes = rng.integers(2, 30, size=n_imp)
    imp = np.repeat(np.arange(n_imp), sizes)
    scores = rng.normal(size=imp.shape[0]).astype(np.float32)
    scores[5] = scores[6]                                        # a tie inside one impression (stable sort matters)
    labels = (rng.random(imp.shape[0]) < 0.2).astype(np.int64)
    first = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    labels[first] = 1
    labels[first + 1] = 0
    sub = [[] for _ in range(n_imp)]
    for i, k in enumerate(imp):
        sub[k].append([float(scores[i]), len(sub[k])])
    res, truth = io.StringIO(), io.StringIO()
    for i, s in enumerate(sub):
        s.sort(key=lambda x: x[0], reverse=True)
        r = [0] * len(s)
        for j in range(len(s)):
            r[s[j][1]] = j + 1
        res.write(('' if i == 0 else '\n') + str(i + 1) + ' ' + str(r).replace(' ', ''))
        lab = labels[imp == i].tolist()
        truth.write(('' if i == 0 else '\n') + str(i + 1) + ' ' + str(lab).replace(' ', ''))
    res.seek(0); truth.seek(0)
    m = ev.scoring(truth, res)
    save_golden(os.path.join(GOLDEN, 'metrics.npz'), imp=imp, scores=scores, labels=labels,
                metrics=np.array(m, dtype=np.float64))
    print('metrics', m)


def cnn_inputs(method):
    cfg = synth.make_text_config(cnn_method=method, cnn_kernel_num=384 if method == 'group3' else 400)
    sd = synth.make_cnn_state_dict(cfg, seed=6)
    tok, mask = synth.make_titles(cfg, 24, seed=3)
    return cfg, sd, tok.view(4, 6, -1), mask.view(4, 6, -1)


def make_cnn_cases():
    """newsEncoders.CNN of the unmodified reference (eval mode), cnn_method naive and group3 (group5 cannot run in the
    reference: layers.py:43-48 concatenates its padding column along the channel dimension)."""
    import importlib
    import pickle
    import tempfile
    for method in ('naive', 'group3'):
        cfg, sd, tok, mask = cnn_inputs(method)
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as tmp:
            os.chdir(tmp)
            try:
                with open('word_embedding-%s-%s-%s-%s.pkl' % (cfg.word_threshold, cfg.word_embedding_dim, cfg.max_title_length,
                                                               cfg.dataset), 'wb') as f:
                    pickle.dump(torch.zeros(cfg.vocabulary_size, cfg.word_embedding_dim), f)
                ne = importlib.import_module('newsEncoders')
                payload = {'meta': np.frombuffer(json.dumps({('w:' + k): sha(v.numpy()) for k, v in sd.items()} |
                                                            {'x:title_text': sha(tok.numpy()), 'x:title_mask': sha(mask.numpy())}).encode(),
                                                 dtype=np.uint8)}
                for tag, dt in (('ref32_', torch.float32), ('ref64_', torch.float64)):
                    m = ne.CNN(cfg)
                    m.load_state_dict(sd)
                    m = m.to(dt).eval()
                    with torch.no_grad():
                        payload[tag + 'news'] = m(tok, mask.to(dt)).numpy()
            finally:
                os.chdir(cwd)
        save_golden(os.path.join(GOLDEN, 'news_encoder_cnn_%s.npz' % method), **payload)
        print('news_encoder_cnn', method, payload['ref32_news'].shape)


if __name__ == '__main__':
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(1)   # fixed reduction partitioning inside MKL/ATen -> reproducible fp32 vectors
    ge, layers, ev, sag = load_reference()
    which = sys.argv[1:] or ['encoder', 'ablation', 'msa', 'cnn', 'sag', 'metrics']
    if 'encoder' in which:
        make_encoder_cases(ge)
    if 'ablation' in which:
        make_ablation_cases(ge)
    if 'msa' in which:
        make_msa_case()
    if 'cnn' in which:
        make_cnn_cases()
    if 'sag' in which:
        make_sag_case(sag)
    if 'metrics' in which:
        make_metric_case(ev)
