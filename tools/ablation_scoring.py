"""Scoring speed of DIGAT and the five ablation encoders: the resident driver against the per-batch ``inference`` loop.

For one workload (bench.build_workload; each encoder gets synth.make_ablation_state_dict weights, DIGAT the bench's) it
times, per encoder:
* ``resident``: scoring.evaluate_resident over the WHOLE corpus (4096-pair batches, de-duplicated user graphs, the
  encoder's per-news cache, on-GPU ranking and metrics; the cache is built before the timed passes);
* ``loop``: what a user of ``encoder.inference()`` runs today -- per 4096-pair batch, gather the seven inputs of reference
  util.py:56-68 from the resident tables (the library's gather kernels and index_select) and call ``inference`` with
  the cached initial context, no sharing between the pairs of an impression -- over the first LOOP_BATCHES batches.
The two paths alternate for ROUNDS rounds in one process after a warm-up; the best round of each is reported.  The
card's name and power limit are read in the same process.

    python tools/ablation_scoring.py --workload mind_small_dev_n3_L3 --out profiles/r4_ablation_scoring_n3_L3.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ROUNDS = 3
BATCH = 4096
LOOP_BATCHES = 40
KINDS = ('DIGAT', 'wo_SA', 'Seq_SA', 'wo_interaction', 'news_graph_wo_inter', 'user_graph_wo_inter')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else ''


def initial_context_table(enc, scorer, chunk=1024):
    """The per-news context the ``inference`` loop reads (reference util.py:37-50), through the public entry points."""
    fn = getattr(enc, 'compute_news_sequence_context', None) or enc.compute_news_graph_context    # Seq_SA: util.py:48
    out = torch.empty((scorer.n_news, scorer.D), device=scorer.dev, dtype=torch.float32)
    for lo in range(0, scorer.n_news, chunk):
        hi = min(lo + chunk, scorer.n_news)
        ids = torch.arange(lo, hi, device=scorer.dev, dtype=torch.int32)
        out[lo:hi] = fn(scorer.gather_sag(ids), scorer.news_mask[lo:hi])
    return out


def inference_loop(enc, scorer, beh, news, c0_table):
    from digat_b200.model import logits
    out = []
    with torch.no_grad():
        for s in range(0, beh.shape[0], BATCH):
            b, nw = beh[s:s + BATCH], news[s:s + BATCH]
            Xn = scorer.gather_sag(nw.to(torch.int32))
            hist = scorer.history.index_select(0, b)
            Xh = scorer.gather_rows(scorer.table, hist.reshape(-1)).view(b.shape[0], hist.shape[1], scorer.D)
            c0 = None if c0_table is None else c0_table.index_select(0, nw)
            cn, cu = enc.inference(Xn, scorer.news_graph.index_select(0, nw), scorer.news_mask.index_select(0, nw), Xh,
                                   scorer.user_graph.index_select(0, b), scorer.cmask.index_select(0, b),
                                   scorer.cidx.index_select(0, b), c0)
            out.append(logits(cn, cu))
    return out


def run_kind(kind, cfg, sd_digat, corpus):
    from digat_b200 import scoring, synth
    from digat_b200.ablation_encoders import ENCODERS
    enc = ENCODERS[kind](cfg, 400)
    enc.load_state_dict(sd_digat if kind == 'DIGAT' else synth.make_ablation_state_dict(kind, cfg, seed=0))
    enc = enc.cuda().eval()
    scorer = scoring.Scorer(enc, corpus, 'cuda:0')
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    scorer.cache_news_context()
    torch.cuda.synchronize()
    cache_s = time.perf_counter() - t0
    c0_table = None if kind == 'wo_SA' else initial_context_table(enc, scorer)
    n_pairs = int(corpus.pair_behavior.shape[0])
    n_loop = min(n_pairs, LOOP_BATCHES * BATCH)
    beh = torch.from_numpy(corpus.pair_behavior[:n_loop]).cuda().long()
    news = torch.from_numpy(corpus.pair_news[:n_loop]).cuda().long()
    # warm-up: every shape of both paths
    warm = [(beh[s:s + BATCH], news[s:s + BATCH]) for s in range(0, 2 * BATCH, BATCH)]
    scoring.score_resident_batches(scorer, warm)
    inference_loop(enc, scorer, beh[:2 * BATCH], news[:2 * BATCH], c0_table)
    torch.cuda.synchronize()
    times = {'resident': [], 'loop': []}
    for _ in range(ROUNDS):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = scoring.evaluate_resident(scorer, corpus, batch_size=BATCH, on_single_class='skip')
        torch.cuda.synchronize()
        times['resident'].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        loop = inference_loop(enc, scorer, beh, news, c0_table)
        torch.cuda.synchronize()
        times['loop'].append(time.perf_counter() - t0)
    scorer.check_index_errors()
    loop = torch.cat(loop)
    agree = (res['scores'][:n_loop] - loop).abs().max().item() / max(loop.abs().max().item(), 1e-30)
    rep = {
        'encoder': type(enc).__name__, 'pairs': n_pairs, 'loop_pairs': n_loop, 'cache_build_s': cache_s,
        'cache_shape': None if scorer.c_n0 is None else list(scorer.c_n0.shape),
        'seconds': times,
        'pairs_per_s': {'resident': n_pairs / min(times['resident']), 'loop': n_loop / min(times['loop'])},
        'metrics': dict(zip(('auc', 'mrr', 'ndcg5', 'ndcg10'), res['metrics'])),
        'max_rel_diff_resident_vs_loop': agree,
    }
    rep['speedup'] = rep['pairs_per_s']['resident'] / rep['pairs_per_s']['loop']
    print(json.dumps({kind: rep['pairs_per_s'], 'speedup': rep['speedup']}), flush=True)
    return rep


def main():
    import bench
    ap = argparse.ArgumentParser()
    ap.add_argument('--workload', default='mind_small_dev_n3_L3', choices=sorted(bench.WORKLOADS))
    ap.add_argument('--out', default=None)
    ap.add_argument('--kinds', nargs='+', default=list(KINDS), choices=KINDS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('ablation_scoring.py needs a CUDA device')
    cfg, sd, corpus = bench.build_workload(args.workload)
    result = {'card': card(), 'workload': args.workload, 'batch': BATCH, 'rounds': ROUNDS, 'best_of_rounds': True,
              'loop_batches': LOOP_BATCHES,
              'encoders': {k: run_kind(k, cfg, sd, corpus) for k in args.kinds}}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
