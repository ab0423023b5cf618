"""The scoring driver (digat_b200/scoring.py) over the five ablation encoders (wo_SA, Seq_SA, wo_interaction,
news_graph_wo_inter, user_graph_wo_inter): each encoder's own scoring schedule (``_encode``), per-news cache
(``_news_cache``) and per-behaviour user stacks, against the CPU oracle (oracle/digat_oracle.py::ablation_inference, the
restatement of reference graphEncoders.py:201-842) and against the encoder's own ``inference``.

* the benchmarked path: two 4096-pair steps of each bench workload through ``score_resident_batches`` and
  ``score_host_batches`` (bit-identical), 256 sampled pairs against the fp32 and fp64 oracle;
* de-duplication is exact (``share_user_graphs`` on / off bit-identical), the scores equal ``inference`` to fp32 accuracy,
  and new weights rebuild the per-news cache;
* ``evaluate_resident`` metrics equal those of the per-batch ``inference`` loop, on one and on two shards;
* errors: out-of-range category ids, encoders without a scoring schedule, BF16 projections."""
import functools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import digat_oracle as O
from tests.helpers import ABLATION_KINDS, err_stats, fmt_stats, rel_err

gpu = pytest.mark.gpu
ORDER = ('news_graph_embeddings', 'news_graph', 'news_graph_mask', 'user_news_embedding', 'user_graph',
         'user_category_mask', 'user_category_indices')
LOGIT_TOL = 1e-5          # fp32 click logits within 1e-5 relative, max-norm (as tests/test_gpu_benchpaths.py)
COND_TOL = 1e-5           # per-logit error relative to sum_d |c_n[d] * c_u[d]|
WORKLOADS = ('mind_small_dev_n3_L3', 'mind_small_dev_n5_L3', 'wide_n8_L7')


def _encoder(kind, cfg, sd):
    """The encoder as Model(config) builds it from the graph_encoder string (reference model.py:18-31)."""
    from digat_b200.model import Model
    model = Model(SimpleNamespace(**dict(vars(cfg), graph_encoder=kind)), 400)
    model.graph_encoder.load_state_dict(sd)
    return model.graph_encoder.cuda().eval()


def _small(kind, seed=0, n_beh=40, L=3):
    from digat_b200 import synth
    cfg = synth.make_config(SAG_neighbors=3, SAG_hops=2, graph_depth=L, graph_encoder=kind)
    sd = synth.make_ablation_state_dict(kind, cfg, seed=seed)
    corpus = synth.make_corpus(cfg, n_news=500, n_behaviors=n_beh, mean_candidates=6.0, seed=seed + 1)
    return cfg, sd, corpus


@functools.lru_cache(maxsize=1)
def _workload(name):
    import bench
    cfg, _, corpus = bench.build_workload(name)
    return cfg, corpus


def _initial_context(enc, kind, X, mask):
    """The cached context each encoder's ``inference`` reads (reference util.py:39-50)."""
    if kind == 'wo_SA':
        return None
    if kind == 'Seq_SA':
        return enc.compute_news_sequence_context(X, mask)
    return enc.compute_news_graph_context(X, mask)


def _oracle_logits(kind, sd, corpus, ids, dtype=torch.float32):
    from digat_b200 import synth
    P = O.cast_params(sd, dtype)
    out, terms = [], []
    with torch.no_grad():
        for s in range(0, len(ids), 64):
            b = synth.make_batch(corpus, ids[s:s + 64])
            a = [b[k].to(dtype) if b[k].is_floating_point() else b[k] for k in ORDER]
            c0 = None if kind == 'wo_SA' else O.news_graph_context(P, a[0], a[2])   # Seq_SA: the same arithmetic
            cn, cu = O.ablation_inference(kind, P, *a, c0)
            out.append(O.logits(cn, cu))
            terms.append((cn * cu).abs().sum(1))
    return torch.cat(out).numpy(), torch.cat(terms).numpy()


def _inference_loop(enc, kind, corpus, batch_size):
    """Scores of the per-batch loop: the seven gathered inputs of reference util.py:56-68, then ``inference``."""
    from digat_b200 import synth
    from digat_b200.model import logits
    n = corpus.pair_behavior.shape[0]
    out = []
    with torch.no_grad():
        for s in range(0, n, batch_size):
            b = {k: v.cuda() for k, v in synth.make_batch(corpus, np.arange(s, min(s + batch_size, n))).items()}
            c0 = _initial_context(enc, kind, b['news_graph_embeddings'], b['news_graph_mask'])
            out.append(logits(*enc.inference(*[b[k] for k in ORDER], c0)))
    enc.check_index_errors()
    return torch.cat(out).cpu().numpy()


@gpu
@pytest.mark.parametrize('workload,kind', [(w, k) for w in WORKLOADS for k in ABLATION_KINDS])
def test_benchmarked_path_matches_oracle(workload, kind):
    from digat_b200 import scoring, synth
    BATCH, STEPS, SAMPLE = 4096, 2, 256
    cfg, corpus = _workload(workload)
    sd = synth.make_ablation_state_dict(kind, cfg, seed=3)
    scorer = scoring.Scorer(_encoder(kind, cfg, sd), corpus, 'cuda:0')
    scorer.cache_news_context()
    beh = torch.from_numpy(corpus.pair_behavior[:BATCH * STEPS]).cuda()
    news = torch.from_numpy(corpus.pair_news[:BATCH * STEPS]).cuda()
    res = torch.cat(scoring.score_resident_batches(
        scorer, ((beh[s * BATCH:(s + 1) * BATCH], news[s * BATCH:(s + 1) * BATCH]) for s in range(STEPS))))
    host = [scoring.host_batch(corpus, np.arange(s * BATCH, (s + 1) * BATCH), pin=True) for s in range(STEPS)]
    hst = torch.cat(scoring.score_host_batches(scorer, host))
    torch.cuda.synchronize()
    scorer.check_index_errors()
    assert res.shape == (BATCH * STEPS,) and bool(torch.isfinite(res).all())
    assert torch.equal(res, hst)                          # both drivers run the same rows through the same kernels
    rng = np.random.Generator(np.random.PCG64(17))
    ids = np.sort(rng.choice(BATCH * STEPS, size=SAMPLE, replace=False))
    ref32, _ = _oracle_logits(kind, sd, corpus, ids, torch.float32)
    ref64, terms64 = _oracle_logits(kind, sd, corpus, ids, torch.float64)
    got = res.cpu().numpy()[ids]
    s32, s64, sref = err_stats(got, ref32, terms64), err_stats(got, ref64, terms64), err_stats(ref32, ref64, terms64)
    print('\n%s %s, %d of %d pairs, logits vs oracle fp32: %s\n    vs fp64: %s\n    oracle fp32 vs fp64: %s'
          % (workload, kind, SAMPLE, BATCH * STEPS, fmt_stats(s32), fmt_stats(s64), fmt_stats(sref)))
    assert s32['max_norm'] < LOGIT_TOL and s64['max_norm'] < LOGIT_TOL, (s32, s64)
    assert s32['cond'] < COND_TOL and s64['cond'] < COND_TOL, (s32, s64)


@gpu
@pytest.mark.parametrize('kind', ABLATION_KINDS)
def test_sharing_inference_and_cache_rebuild(kind):
    from digat_b200 import scoring, synth
    cfg, sd, corpus = _small(kind)
    enc = _encoder(kind, cfg, sd)
    scorer = scoring.Scorer(enc, corpus, 'cuda:0')
    n = corpus.pair_behavior.shape[0]
    beh = torch.from_numpy(corpus.pair_behavior).cuda()
    news = torch.from_numpy(corpus.pair_news).cuda()
    shared = scorer.score_resident(beh, news, share_user_graphs=True)
    plain = scorer.score_resident(beh, news, share_user_graphs=False)
    hb = scoring.host_batch(corpus, np.arange(n))
    host_shared = scorer.score_host_batch(*hb, share_user_graphs=True)
    host_plain = scorer.score_host_batch(*hb, share_user_graphs=False)
    scorer.check_index_errors()
    # per-behaviour user stacks and the per-news cache re-use the same rows through the same kernels: bit-identical
    assert torch.equal(shared, plain)
    assert torch.equal(host_shared, host_plain) and torch.equal(host_shared, shared)
    # the encoder's own inference on the same batch
    b = {k: v.cuda() for k, v in synth.make_batch(corpus, np.arange(n)).items()}
    from digat_b200.model import logits
    with torch.no_grad():
        c0 = _initial_context(enc, kind, b['news_graph_embeddings'], b['news_graph_mask'])
        inf = logits(*enc.inference(*[b[k] for k in ORDER], c0))
    assert rel_err(shared.cpu().numpy(), inf.cpu().numpy()) < 1e-5
    ids = np.arange(n)
    ref, _ = _oracle_logits(kind, sd, corpus, ids)
    assert rel_err(shared.cpu().numpy(), ref) < LOGIT_TOL
    # new weights: the packed weights and with them the per-news cache are rebuilt before the next batch
    sd2 = synth.make_ablation_state_dict(kind, cfg, seed=10)
    enc.load_state_dict(sd2)
    again = scorer.score_resident(beh, news).cpu().numpy()
    ref2, _ = _oracle_logits(kind, sd2, corpus, ids)
    assert rel_err(again, ref2) < LOGIT_TOL, rel_err(again, ref2)
    assert rel_err(ref2, ref) > 1e-2                   # the two weight sets do score differently


@gpu
@pytest.mark.parametrize('kind', ABLATION_KINDS)
def test_evaluate_resident_matches_the_inference_loop(kind):
    import dataclasses
    from digat_b200 import evaluate, scoring
    cfg, sd, corpus = _small(kind, seed=5, n_beh=300)
    counts = np.bincount(corpus.pair_behavior, minlength=300)
    sel = counts[corpus.pair_behavior] >= 2                                  # AUC needs both classes
    corpus = dataclasses.replace(corpus, pair_behavior=corpus.pair_behavior[sel], pair_news=corpus.pair_news[sel],
                                 labels=corpus.labels[sel])
    enc = _encoder(kind, cfg, sd)
    scorer = scoring.Scorer(enc, corpus, 'cuda:0')
    out = scoring.evaluate_resident(scorer, corpus, batch_size=512)
    loop = _inference_loop(enc, kind, corpus, 512)
    scores = out['scores'].cpu().numpy()
    assert rel_err(scores, loop) < 1e-5
    imp = np.cumsum(np.concatenate([[0], np.diff(corpus.pair_behavior) != 0]))
    labels = [corpus.labels[imp == i].tolist() for i in range(int(imp[-1]) + 1)]
    m_loop = evaluate.metrics(evaluate.rank_lists(loop, imp), labels)
    assert np.allclose(out['metrics'], m_loop, atol=1e-4), (out['metrics'], m_loop)
    # two shards of whole impressions, run in turn: concatenated ranks equal the single-shard ranks
    parts = [scoring.evaluate_resident(scorer, corpus, batch_size=512, rank=r, world_size=2) for r in range(2)]
    assert torch.equal(torch.cat([p['ranks'] for p in parts]), out['ranks'])


@gpu
@pytest.mark.parametrize('kind', ABLATION_KINDS)
def test_out_of_range_category_index_is_reported(kind):
    from digat_b200 import scoring
    cfg, sd, corpus = _small(kind, n_beh=8)
    scorer = scoring.Scorer(_encoder(kind, cfg, sd), corpus, 'cuda:0')
    scorer.cidx[0, 0] = 10 ** 6                                            # corrupt one history slot of behaviour 0
    beh = torch.zeros(4, dtype=torch.int64, device='cuda')
    news = torch.tensor([1, 2, 3, 4], device='cuda')
    scorer.score_resident(beh, news)
    with pytest.raises(RuntimeError, match='user_category_indices'):
        scorer.check_index_errors()


@gpu
@pytest.mark.parametrize('kind', ABLATION_KINDS)
def test_ablation_scorer_still_refuses_bf16(kind):
    from digat_b200 import scoring
    cfg, sd, corpus = _small(kind, n_beh=8)
    enc = _encoder(kind, cfg, sd)
    enc.projection_precision = 'bf16'
    scorer = scoring.Scorer(enc, corpus, 'cuda:0')
    beh = torch.zeros(4, dtype=torch.int64, device='cuda')
    news = torch.tensor([1, 2, 3, 4], device='cuda')
    with pytest.raises(RuntimeError, match='bf16'):
        scorer.score_resident(beh, news)


def test_scorer_refuses_encoders_without_a_scoring_schedule():
    """Checked before anything touches the device: runs without a GPU."""
    from digat_b200 import scoring, synth
    from digat_b200.ablation_encoders import _AblationEncoder
    from digat_b200.graphEncoders import GraphEncoder

    class PlainEncoder(GraphEncoder):
        pass

    class CustomAblation(_AblationEncoder):
        NEWS_LAYER = 'gat'

    cfg = synth.make_config()
    for enc in (PlainEncoder(cfg, 400), CustomAblation(cfg, 400)):
        with pytest.raises(RuntimeError, match='supported encoders: DIGAT, wo_SA'):
            scoring.Scorer(enc, None, 'cpu')
