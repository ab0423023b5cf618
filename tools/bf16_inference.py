"""Speed and ranking metrics of DIGAT.projection_precision = 'bf16' against the fp32 default (DESIGN.md section 4.8).

For each workload (bench.build_workload: BASELINE.json configs[1] and configs[3]) it runs scoring.evaluate_resident over
the WHOLE corpus in both modes, alternating fp32 / bf16 for ROUNDS rounds in one process, and reports pairs/s per mode,
the four metric deltas and the largest logit difference.  A separate profiled pass over the first PROFILE_PAIRS pairs
times every call of digat_linear_tf32x3 / digat_linear_bf16 with CUDA events (digat_b200._lib.start_profile) and
turns the GEMM shapes into FLOP/s.  The card's name and power limit are read in the same process.

    python tools/bf16_inference.py [--out profiles/r3_bf16_inference.json] [--workloads mind_small_dev_n3_L3 wide_n8_L7]
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
PROFILE_PAIRS = 40 * BATCH
GEMMS = ('digat_linear_tf32x3', 'digat_linear_bf16')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else ''


def gemm_profile(scorer, corpus, mode):
    from digat_b200 import _lib, scoring
    scorer.enc.projection_precision = mode
    beh = torch.from_numpy(corpus.pair_behavior[:PROFILE_PAIRS]).cuda()
    news = torch.from_numpy(corpus.pair_news[:PROFILE_PAIRS]).cuda()
    batches = [(beh[s:s + BATCH], news[s:s + BATCH]) for s in range(0, PROFILE_PAIRS, BATCH)]
    scoring.score_resident_batches(scorer, batches[:2])                    # warm every shape
    torch.cuda.synchronize()
    w = scorer.enc._weights()
    proj = {pw.wb.data_ptr() if pw.wb is not None else pw.hi.data_ptr()    # the GEMMs the mode moves: Wcat, featureAffine
            for k, pw in w.items() if (isinstance(k, tuple) and k[-1] == 'Wcat') or k == 'fa_W'}
    _lib.start_profile()
    scoring.score_resident_batches(scorer, batches)
    torch.cuda.synchronize()
    rec = _lib.stop_profile()
    out = {}
    for name, args, ms in rec:
        if name not in GEMMS:
            continue
        i = 8 if name == 'digat_linear_tf32x3' else 7                      # position of M in the C signature
        M, N, K = args[i:i + 3]
        key = '%s %s N=%d' % (name, 'projection' if args[2] in proj else 'other', N)
        e = out.setdefault(key, {'calls': 0, 'ms': 0.0, 'flop': 0.0, 'rows': 0})
        e['calls'] += 1
        e['ms'] += ms
        e['flop'] += 2.0 * M * N * K
        e['rows'] += M
    for e in out.values():
        e['tflops'] = e['flop'] / (e['ms'] * 1e-3) / 1e12
        e['ms_per_call'] = e['ms'] / e['calls']
        e['ms'] = round(e['ms'], 3)
    return out


def run(workload):
    import bench
    from digat_b200 import scoring
    from digat_b200.graphEncoders import DIGAT
    cfg, sd, corpus = bench.build_workload(workload)
    enc = DIGAT(cfg, 400)
    enc.load_state_dict(sd)
    enc = enc.cuda().eval()
    scorer = scoring.Scorer(enc, corpus, 'cuda:0', build_user_graphs_on_device=True)
    scorer.cache_news_context()
    n_pairs = int(corpus.pair_behavior.shape[0])
    times = {'fp32': [], 'bf16': []}
    res = {}
    for r in range(ROUNDS + 1):                                             # round 0 warms both modes up
        for mode in ('fp32', 'bf16'):
            enc.projection_precision = mode
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = scoring.evaluate_resident(scorer, corpus, batch_size=BATCH, on_single_class='skip')
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if r > 0:
                times[mode].append(dt)
            res[mode] = out
    d = [b - a for a, b in zip(res['fp32']['metrics'], res['bf16']['metrics'])]
    rep = {
        'workload': workload, 'pairs': n_pairs, 'batch': BATCH, 'rounds': ROUNDS,
        'seconds': times,
        'pairs_per_s': {m: n_pairs / min(t) for m, t in times.items()},
        'pairs_per_s_median': {m: n_pairs / sorted(t)[len(t) // 2] for m, t in times.items()},
        'metrics': {m: dict(zip(('auc', 'mrr', 'ndcg5', 'ndcg10'), res[m]['metrics'])) for m in res},
        'metric_delta_bf16_minus_fp32': dict(zip(('auc', 'mrr', 'ndcg5', 'ndcg10'), d)),
        'max_abs_logit_diff': float((res['bf16']['scores'] - res['fp32']['scores']).abs().max()),
        'max_abs_logit_fp32': float(res['fp32']['scores'].abs().max()),
        'gemm_profile': {m: gemm_profile(scorer, corpus, m) for m in ('fp32', 'bf16')},
    }
    rep['speedup'] = rep['pairs_per_s']['bf16'] / rep['pairs_per_s']['fp32']
    enc.projection_precision = 'fp32'
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--workloads', nargs='+', default=['mind_small_dev_n3_L3', 'wide_n8_L7'])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bf16_inference.py needs a CUDA device')
    result = {'card': card(), 'profile_pairs': PROFILE_PAIRS, 'workloads': [run(w) for w in args.workloads]}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
