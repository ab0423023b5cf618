"""BF16 node projections at inference (DIGAT.projection_precision = 'bf16', digat_linear_bf16, DESIGN.md section 4.8):

* the GEMM against its own contract: fp64 product of the RNE-rounded operands, row scatter and row-range splits
  bit-identical to the dense call;
* one layer against the oracle with the same operands rounded (oracle._lin replaced for the Wcat / featureAffine weights);
* the encoder against the exact fp64 oracle (golden cases x64, sampled pairs of the three bench workloads), gate 2e-3;
* AUC / MRR / nDCG@5 / nDCG@10 on the full MIND-small-dev-sized corpus within 1e-4 of the fp32 mode;
* the invariants of the fp32 mode (shared vs expanded user graphs, pruning on / off, both scoring drivers) hold;
* the training path and the ablation encoders are not affected / refuse the mode."""
import numpy as np
import pytest
import torch

from oracle import digat_oracle as O
from tests.helpers import (ABLATION_KINDS, CASES, ablation_inputs, case_inputs, check_hashes, err_stats, fmt_stats,
                           load_golden, rel_err)

ORDER = ('news_graph_embeddings', 'news_graph', 'news_graph_mask', 'user_news_embedding', 'user_graph',
         'user_category_mask', 'user_category_indices')
GEMM_TOL = 1e-5           # kernel vs fp64 product of the bf16-rounded operands, relative to max|C|
LAYER_TOL = 1e-5          # one layer vs the oracle with the same operands rounded
LOGIT_TOL = 2e-3          # logits vs the exact fp64 oracle, max-norm
METRIC_TOL = 1e-4         # AUC / MRR / nDCG: the only tolerance the reference states (README.md:64)
REPLICAS = 64


def _rounded_ref(A, W, bias=None, gbias=None, group_rows=1, group_col0=0):
    ref = A.to(torch.bfloat16).double() @ W.to(torch.bfloat16).double().t()
    if bias is not None:
        ref += bias.double()
    if gbias is not None:
        g = torch.arange(A.shape[0], device=A.device) // group_rows
        ref[:, group_col0:group_col0 + gbias.shape[1]] += gbias.double()[g]
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize('N', [1200, 400])
@pytest.mark.parametrize('M', [1, 127, 300, 20000, 136000])
def test_linear_bf16_against_rounded_operands(M, N):
    from digat_b200 import _lib
    from digat_b200.graphEncoders import PackedWeight, linear
    g = torch.Generator().manual_seed(M * 7 + N)
    K = 400
    W = (torch.randn(N, K, generator=g) * 0.05).cuda()
    Wp = PackedWeight(W, bf16=True)
    bias = torch.randn(N, generator=g).cuda()
    rows = 68 if N == 1200 else 19
    gbias = torch.randn((M + rows - 1) // rows, 400, generator=g).cuda()
    col0 = 400 if N == 1200 else 0
    X = torch.randn(M, K + 24, generator=g).cuda()                           # strided A: lda = K + 24
    for strided in (False, True):
        A = X[:, :K] if strided else X[:, :K].contiguous()
        for with_bias, with_gb in ((False, False), (True, False), (True, True)):
            kw = dict(group_bias=gbias, group_rows=rows, group_col0=col0) if with_gb else {}
            _lib.start_profile()
            if strided:
                C = linear(A, Wp, bias if with_bias else None, M=M, K=K, lda=K + 24, **kw)
            else:
                C = linear(A, Wp, bias if with_bias else None, **kw)
            torch.cuda.synchronize()
            assert [r[0] for r in _lib.stop_profile()] == ['digat_linear_bf16']   # every M takes the BF16 kernel
            ref = _rounded_ref(A, W, bias if with_bias else None, gbias if with_gb else None, rows, col0)
            err = float((C.double() - ref).abs().max() / ref.abs().max())
            assert err <= GEMM_TOL, (M, N, strided, with_bias, with_gb, err)


@pytest.mark.gpu
@pytest.mark.parametrize('M_full,N,frac', [(68 * 700, 1200, 0.5), (68 * 3, 1200, 0.5), (19 * 500, 400, 0.7)])
def test_linear_bf16_row_scatter_and_row_ranges_bit_identical(M_full, N, frac):
    from digat_b200.graphEncoders import PackedWeight, linear
    g = torch.Generator().manual_seed(M_full + N)
    K, rows_per_group = 400, 68 if N == 1200 else 19
    col0 = 400 if N == 1200 else 0
    X = torch.randn(M_full, K, generator=g).cuda()
    W = PackedWeight((torch.randn(N, K, generator=g) * 0.05).cuda(), bf16=True)
    bias = torch.randn(N, generator=g).cuda()
    gbias = torch.randn(M_full // rows_per_group, 400, generator=g).cuda()
    kw = dict(group_bias=gbias, group_rows=rows_per_group, group_col0=col0)
    full = linear(X, W, bias, **kw)
    keep = torch.rand(M_full, generator=g) < frac
    keep[:rows_per_group] = False                                            # a whole group without rows
    rows = keep.nonzero().squeeze(1).to(torch.int32).cuda()
    A = X[rows.long()].contiguous()
    out = torch.full((M_full, N), 7.0, device='cuda')
    linear(A, W, bias, out=out, c_rows=rows, **kw)
    # one M as two calls over different row ranges (the second starts mid-tile): tile position does not matter
    m1 = rows_per_group * (M_full // rows_per_group // 3)
    two = torch.empty_like(full)
    linear(X[:m1], W, bias, out=two[:m1], group_bias=gbias[:m1 // rows_per_group], group_rows=rows_per_group,
           group_col0=col0)
    linear(X[m1:], W, bias, out=two[m1:], group_bias=gbias[m1 // rows_per_group:], group_rows=rows_per_group,
           group_col0=col0)
    torch.cuda.synchronize()
    k = keep.cuda()
    assert torch.equal(out[k], full[k])
    assert bool((out[~k] == 7.0).all())
    assert torch.equal(two, full)


def _encoder(cfg, sd, precision='bf16'):
    from digat_b200.graphEncoders import DIGAT
    m = DIGAT(cfg, 400)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    m.projection_precision = precision
    return m


def _round_operands_lin(P, names):
    """oracle._lin with A and W rounded to bf16 (RNE) for the weights listed, exact otherwise."""
    ids = {id(P[k]) for k in names}
    exact = O._lin

    def lin(x, w, b=None):
        if id(w) in ids:
            return exact(x.to(torch.bfloat16).to(x.dtype), w.to(torch.bfloat16).to(w.dtype), b)
        return exact(x, w, b)
    return lin


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['default_n3_L3', 'wide_n8_L7'])
def test_one_layer_against_oracle_with_rounded_projections(name, monkeypatch):
    cfg, sd, corpus, batch = case_inputs(name)
    m = _encoder(cfg, sd)
    bb = {k: v.repeat(REPLICAS, *([1] * (v.dim() - 1))) for k, v in batch.items()}
    b = {k: v.cuda() for k, v in bb.items()}
    P = O.cast_params(sd, torch.float64)
    with torch.no_grad():
        c_n0 = m.compute_news_graph_context(b['news_graph_embeddings'], b['news_graph_mask'])
        Xu = torch.cat([b['user_news_embedding'], m.topic_node_embedding.unsqueeze(0).expand(c_n0.shape[0], -1, -1)], 1)
        c_u0 = m.compute_user_graph_context(Xu, b['user_category_mask'], b['user_category_indices'], c_n0)
    names = ['featureAffine.weight'] + ['%s_graph_attention_%s.%d.weight' % (g, f, i) for g in ('news', 'user')
                                        for f in ('W', 'ffn1', 'ffn2') for i in range(cfg.graph_depth)]
    monkeypatch.setattr(O, '_lin', _round_operands_lin(P, names))
    d = lambda t: t.cpu().double()                                           # noqa: E731
    for i in range(cfg.graph_depth):                                         # each layer's weights on the same operands
        with torch.no_grad():
            Yn = m.compute_news_graph_embeddings(i, b['news_graph_embeddings'], b['news_graph'], c_u0)
            Yu = m.compute_user_graph_embeddings(i, Xu, b['user_graph'], c_n0)
        rn = O.graph_layer(P, 'news', i, d(b['news_graph_embeddings']), bb['news_graph'], d(c_u0))
        ru = O.graph_layer(P, 'user', i, d(Xu), bb['user_graph'], d(c_n0))
        en, eu = rel_err(Yn.cpu().numpy(), rn.numpy()), rel_err(Yu.cpu().numpy(), ru.numpy())
        print('\n%s layer %d: news %.2e, user %.2e' % (name, i, en, eu))
        assert en < LAYER_TOL and eu < LAYER_TOL, (i, en, eu)


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(CASES))
def test_golden_cases_replicated_against_fp64_oracle(name):
    from digat_b200 import _lib
    from digat_b200.model import logits
    cfg, sd, corpus, batch = case_inputs(name)
    z, meta = load_golden(name)
    check_hashes(meta, sd, batch)
    m = _encoder(cfg, sd)
    B = batch['news_graph'].shape[0]
    bb = {k: v.cuda().repeat(REPLICAS, *([1] * (v.dim() - 1))) for k, v in batch.items()}
    args = [bb[k] for k in ORDER]
    _lib.start_profile()
    with torch.no_grad():
        c_n0 = m.compute_news_graph_context(bb['news_graph_embeddings'], bb['news_graph_mask'])
        lg = logits(*m.inference(*args, c_n0))
        lf = logits(*m.forward(*args))
    torch.cuda.synchronize()
    names = [r[0] for r in _lib.stop_profile()]
    assert 'digat_linear_bf16' in names
    # c_n0 uses none of the BF16 projections: it is the fp32 mode's, to the bit
    ref_c_n0 = _encoder(cfg, sd, 'fp32').compute_news_graph_context(bb['news_graph_embeddings'], bb['news_graph_mask'])
    assert torch.equal(c_n0, ref_c_n0)
    ref64 = z['ref64_logits']
    terms = np.abs(z['ref64_news_ctx'] * z['ref64_user_ctx']).sum(1)
    for lo in (lg, lf):
        got = lo.cpu().numpy()
        for r in range(REPLICAS):
            s = err_stats(got[r * B:(r + 1) * B], ref64, terms)
            assert s['max_norm'] <= LOGIT_TOL, (r, s)
    s = err_stats(lg.cpu().numpy()[:B], ref64, terms)
    print('\n%s x%d bf16 logits vs fp64 reference: %s (gate max_norm %.0e)' % (name, REPLICAS, fmt_stats(s), LOGIT_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('workload', ['mind_small_dev_n3_L3', 'mind_small_dev_n5_L3', 'wide_n8_L7'])
def test_bench_batch_sampled_against_fp64_oracle(workload):
    import bench
    from digat_b200 import scoring
    from tests.test_gpu_benchpaths import _oracle_logits
    BATCH, STEPS, SAMPLE = 4096, 2, 256
    cfg, sd, corpus = bench.build_workload(workload)
    scorer = scoring.Scorer(_encoder(cfg, sd), corpus, 'cuda:0')
    scorer.cache_news_context()
    beh = torch.from_numpy(corpus.pair_behavior[:BATCH * STEPS]).cuda()
    news = torch.from_numpy(corpus.pair_news[:BATCH * STEPS]).cuda()
    res = torch.cat(scoring.score_resident_batches(
        scorer, ((beh[s * BATCH:(s + 1) * BATCH], news[s * BATCH:(s + 1) * BATCH]) for s in range(STEPS))))
    host = [scoring.host_batch(corpus, np.arange(s * BATCH, (s + 1) * BATCH), pin=True) for s in range(STEPS)]
    hst = torch.cat(scoring.score_host_batches(scorer, host))
    torch.cuda.synchronize()
    scorer.check_index_errors()
    assert bool(torch.isfinite(res).all())
    assert torch.equal(res, hst)                                             # both drivers: same rows, same kernels
    rng = np.random.Generator(np.random.PCG64(17))
    ids = np.sort(rng.choice(BATCH * STEPS, size=SAMPLE, replace=False))
    ref64, terms64 = _oracle_logits(sd, corpus, ids, torch.float64)
    s = err_stats(res.cpu().numpy()[ids], ref64, terms64)
    print('\n%s, %d of %d pairs, bf16 logits vs oracle fp64: %s (gate max_norm %.0e)'
          % (workload, SAMPLE, BATCH * STEPS, fmt_stats(s), LOGIT_TOL))
    assert s['max_norm'] <= LOGIT_TOL, s


@pytest.mark.gpu
def test_full_corpus_metrics_within_1e4_of_fp32():
    import bench
    from digat_b200 import scoring
    cfg, sd, corpus = bench.build_workload('mind_small_dev_n3_L3')
    enc = _encoder(cfg, sd, 'fp32')
    scorer = scoring.Scorer(enc, corpus, 'cuda:0', build_user_graphs_on_device=True)
    scorer.cache_news_context()
    out = {}
    for mode in ('fp32', 'bf16'):
        enc.projection_precision = mode
        out[mode] = scoring.evaluate_resident(scorer, corpus, batch_size=4096, on_single_class='skip')
    d = [b - a for a, b in zip(out['fp32']['metrics'], out['bf16']['metrics'])]
    dl = float((out['bf16']['scores'] - out['fp32']['scores']).abs().max())
    print('\nfull corpus (%d pairs): fp32 %s, bf16 %s, delta (auc, mrr, ndcg5, ndcg10) %s, max |logit diff| %.3e'
          % (out['fp32']['scores'].shape[0], ['%.6f' % v for v in out['fp32']['metrics']],
             ['%.6f' % v for v in out['bf16']['metrics']], ['%+.2e' % v for v in d], dl))
    assert all(abs(v) <= METRIC_TOL for v in d), d


@pytest.mark.gpu
def test_scoring_invariants_hold_in_bf16_mode():
    from tests.test_gpu_scoring import _setup
    cfg, sd, corpus, scorer = _setup(n_beh=50, seed=9)
    scorer.enc.projection_precision = 'bf16'
    beh = torch.from_numpy(corpus.pair_behavior).cuda()
    news = torch.from_numpy(corpus.pair_news).cuda()
    scorer.enc.prune_user_nodes = True
    a = scorer.score_resident(beh, news)
    a2 = scorer.score_resident(beh, news, share_user_graphs=False)
    scorer.enc.prune_user_nodes = False
    b = scorer.score_resident(beh, news)
    b2 = scorer.score_resident(beh, news, share_user_graphs=False)
    assert torch.equal(a, a2) and torch.equal(a, b) and torch.equal(a, b2)
    scorer.enc.projection_precision = 'fp32'
    assert not torch.equal(scorer.score_resident(beh, news), a)              # the mode really switched


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['default_n3_L3', 'wide_n8_L7'])
def test_inference_identical_with_and_without_pruning_in_bf16_mode(name):
    cfg, sd, corpus, batch = case_inputs(name)
    m = _encoder(cfg, sd)
    b = {k: v.cuda().repeat(REPLICAS, *([1] * (v.dim() - 1))) for k, v in batch.items()}
    args = [b[k] for k in ORDER]
    with torch.no_grad():
        c0 = m.compute_news_graph_context(b['news_graph_embeddings'], b['news_graph_mask'])
        m.prune_user_nodes = True
        cn1, cu1 = m.inference(*args, c0)
        m.prune_user_nodes = False
        cn0, cu0 = m.inference(*args, c0)
    assert torch.equal(cn1, cn0) and torch.equal(cu1, cu0)


@pytest.mark.gpu
def test_training_gradients_ignore_the_mode():
    from digat_b200 import _lib
    cfg, sd, corpus, batch = case_inputs('default_n3_L3')
    b = {k: v.cuda().repeat(8, *([1] * (v.dim() - 1))) for k, v in batch.items()}
    grads = {}
    for mode in ('fp32', 'bf16'):
        m = _encoder(cfg, sd, mode)
        _lib.start_profile()
        cn, cu = m(*[b[k] for k in ORDER])
        (cn * cu).sum().backward()
        torch.cuda.synchronize()
        assert 'digat_linear_bf16' not in [r[0] for r in _lib.stop_profile()]
        grads[mode] = [p.grad.clone() for p in m.parameters()]
    assert all(torch.equal(x, y) for x, y in zip(grads['fp32'], grads['bf16']))


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ABLATION_KINDS)
def test_ablation_encoders_refuse_bf16(kind):
    from digat_b200.ablation_encoders import ENCODERS
    cfg, sd, batch = ablation_inputs(kind, 'n3_L2')
    m = ENCODERS[kind](cfg, 400)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    m.projection_precision = 'bf16'
    with torch.no_grad(), pytest.raises(RuntimeError, match='bf16'):
        m.inference(*[batch[k].cuda() for k in ORDER],
                    torch.zeros(batch['news_graph'].shape[0], 400, device='cuda'))


def test_unknown_precision_raises_without_a_gpu():
    from digat_b200 import synth
    from digat_b200.graphEncoders import DIGAT
    m = DIGAT(synth.make_config(SAG_neighbors=3, SAG_hops=2, graph_depth=2), 400)
    assert DIGAT.projection_precision == 'fp32' and m.projection_precision == 'fp32'
    m.projection_precision = 'fp16'
    with pytest.raises(ValueError, match='projection_precision'):
        m._weights()
