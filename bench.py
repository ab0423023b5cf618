#!/usr/bin/env python
"""bench.py -- DIGAT dual-graph encoder: pairs ("impressions") scored per second on synthetic MIND-shaped data.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                     (the reference's CPU algorithm = oracle port, host cores)

A step = one pass of the hot path over one batch of `--batch` (user behaviour, candidate news) pairs of the
synthetic MIND-small-dev-sized corpus (BASELINE.json configs[1]; SURVEY.md section 8d).
  value : pairs/s with the corpus resident in HBM (pair = (behaviour index, news id); gathers + encoder + logits)
  e2e   : pairs/s through scoring.score_host_batches with HOST (pinned) per-pair tensors, H2D + D2H inside the timing
          (both drivers stage batch k+1 on a side stream while batch k is encoded)
  sustained : the same resident path run back to back for >= --sustained seconds (median SM clock / throttle reasons of
          that window) next to the 20-step burst
  train : BASELINE.json configs[2] -- fwd+bwd+clip+Adam on 64 behaviours x 5 candidates per GPU, DDP/NCCL gradient
          all-reduce when N>1: samples/s, per-kernel table, CPU-oracle fwd+bwd baseline (N=1), 1-vs-N gradient equality (N>1)
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D = 400
WORKLOADS = {
    # name: (SAG_neighbors, SAG_hops, graph_depth, n_news, n_behaviors, mean_candidates)
    'mind_small_dev_n3_L3': (3, 2, 3, 65238, 73152, 37.5),       # BASELINE.json configs[1]
    'mind_small_dev_n5_L3': (5, 2, 3, 65238, 73152, 37.5),       # the reference's argparse default (config.py:53)
    'wide_n8_L7': (8, 2, 7, 65238, 73152, 37.5),                 # BASELINE.json configs[3]
    # BASELINE.json configs[4] at FULL size (scale factor 1.0): 161 013 news, 2.37 M behaviours, ~8.8e7 pairs in total.
    # Every rank holds the whole news side and generates + holds only ITS contiguous 1/N shard of the behaviours (their
    # [N_beh,68,68] graphs are built on the device from 200 B/behaviour of category ids).
    'mind_large_8gpu': (3, 2, 3, 161013, 2370000, 37.0),
}
SHARDED_WORKLOADS = ('mind_large_8gpu',)


def algorithmic_bytes_per_pair(n_n, n_u, L, H=50, C=18):
    """B_alg of SURVEY.md section 8(d): layer-granular compulsory HBM traffic of the design."""
    S, T = n_n * n_n + n_u * n_u, n_n + n_u
    b_in = 4 * D * (n_n + H + 1) + S + n_n + (C + 1) + 8 * H + 16
    return L * (4 * D * (9 * T + n_n + H) + S) + b_in


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons while the timed region runs: through NVML in-process (pynvml, two cheap
    queries every 25 ms) when available, else with an `nvidia-smi -lms 100` child process (the recipe's clocks line)."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None
        self.mode = os.environ.get('DIGAT_BENCH_SAMPLER', 'nvml')
        self._stop_flag = False

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        idx = int(vis.split(',')[self.gpu]) if vis and all(x.strip().isdigit() for x in vis.split(',')) else self.gpu
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        bits = [(getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8), 3), (getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40), 4),
                (getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20), 5), (getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4), 6)]
        while not self._stop_flag:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            row = [str(sm), str(mx), '', 'Not Active', 'Not Active', 'Not Active', 'Not Active']
            for bit, col in bits:
                if rs & bit:
                    row[col] = 'Active'
            self.rows.append(row)
            time.sleep(0.025)

    def run(self):
        if self.mode == 'none':
            return
        if self.mode == 'nvml':
            try:
                self._run_nvml()
                return
            except Exception:
                if self.rows:
                    return
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(',')])
        except Exception:
            pass

    def mark(self):
        """Index of the next sample (windows of the sample list: stats(lo, hi))."""
        return len(self.rows)

    def stats(self, lo=0, hi=None):
        rows = self.rows[lo:hi]
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i] == 'Active' for r in rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}

    def stop(self, lo=0, hi=None):
        self._stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        return self.stats(lo, hi)


def build_workload(name, seed=0, rank=0, world=1):
    """-> (config, state_dict, corpus).  Sharded workloads generate only this rank's 1/world of the behaviours (same news
    side on every rank); the others generate the whole corpus and shard the ordered pair list (scoring.shard_range)."""
    from digat_b200 import synth
    N, hops, L, n_news, n_beh, cand = WORKLOADS[name]
    cfg = synth.make_config(SAG_neighbors=N, SAG_hops=hops, graph_depth=L)
    sd = synth.make_state_dict(cfg, D=D, seed=seed)
    if name in SHARDED_WORKLOADS:
        per = (n_beh + world - 1) // world
        mine = max(0, min(per, n_beh - rank * per))
        corpus = synth.make_corpus(cfg, D=D, n_news=n_news, n_behaviors=mine, mean_candidates=cand, seed=seed,
                                   behavior_seed=seed + rank, build_user_graph=False)
    else:
        corpus = synth.make_corpus(cfg, D=D, n_news=n_news, n_behaviors=n_beh, mean_candidates=cand, seed=seed)
    return cfg, sd, corpus


def oracle_pairs_per_second(cfg, sd, corpus, rows, budget_s, steps=None, warmup=2):
    """Times the CPU oracle (port of the reference algorithm, oracle/digat_oracle.py) on `rows` pairs per call."""
    from digat_b200 import synth
    from oracle import digat_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = O.cast_params(sd)
    order = ('news_graph_embeddings', 'news_graph', 'news_graph_mask', 'user_news_embedding', 'user_graph',
             'user_category_mask', 'user_category_indices')
    batch = synth.make_batch(corpus, np.arange(rows))
    args = [batch[k] for k in order]
    with torch.no_grad():
        c_n0 = O.news_graph_context(P, batch['news_graph_embeddings'], batch['news_graph_mask'])
        for _ in range(warmup):
            O.logits(*O.inference(P, *args, c_n0))
        n, t0 = 0, time.perf_counter()
        while True:
            O.logits(*O.inference(P, *args, c_n0))
            n += 1
            el = time.perf_counter() - t0
            if (steps is not None and n >= steps) or (steps is None and el >= budget_s):
                break
    return n * rows / el, el / n, cores, n


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cfg, sd, corpus = build_workload(args.workload)
    rows = 64
    pps, sec, cores, n = oracle_pairs_per_second(cfg, sd, corpus, rows, None, steps=args.steps, warmup=args.warmup)
    sample = '%d calls of DIGAT.inference on %d pairs each (oracle port of reference graphEncoders.py:189-198)' % (n, rows)
    print(json.dumps({
        'impl': 'reference', 'metric': 'impressions_scored_per_sec', 'value': pps, 'unit': 'pairs/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': args.workload, 'rows_per_step': rows, 'device': 'host cpu'},
        'cpu_baseline': {'value': pps, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': pps, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }))


def _dist_env():
    return int(os.environ.get('RANK', '0')), int(os.environ.get('LOCAL_RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))


def _max_over_ranks(ms, world, dev):
    if world == 1:
        return ms
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def _peaks():
    peaks = {}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(pk):
        peaks = json.load(open(pk))
    return (float(peaks.get('hbm_gbs', 6650.0)),
            float(peaks.get('bf16_tflops_sustained', peaks.get('bf16_tflops', 1590.0))),
            'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=4096, help='pairs per step per GPU')
    ap.add_argument('--workload', default='mind_small_dev_n3_L3', choices=list(WORKLOADS))
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-budget', type=float, default=12.0, help='seconds of CPU-oracle timing for cpu_baseline')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--sustained', type=float, default=5.0,
                    help='seconds of back-to-back resident steps for the `sustained` sub-record (0 = skip)')
    ap.add_argument('--no-train', action='store_true', help='score mode: skip the `train` sub-record')
    ap.add_argument('--train-steps', type=int, default=20)
    ap.add_argument('--eager-train', action='store_true',
                    help='train: run the step eagerly instead of replaying it as one CUDA graph')
    ap.add_argument('--mode', default='score', choices=['score', 'train', 'train_tokens'],
                    help="'score' = the headline metric (+ sustained + train sub-records); 'train' = only the training record "
                         "(fwd+bwd(+DDP all-reduce)+clip+Adam step, samples/s) as the line; 'train_tokens' = the same step from "
                         "TOKEN tensors, MSA news encoder included (reference Model.forward, model.py:54-77), eager, one GPU")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="score mode: write the click logits of the last timed step to DIR/logits.npy (float32; "
                         "DIR/logits_rank<r>.npy per rank when N>1), to compare two builds on identical seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'ours' or args.mode != 'score'):
        ap.error('--dump-outputs needs --impl ours --mode score')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    if args.impl == 'reference':
        run_reference_arm(args)
        return

    rank, local_rank, world = _dist_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        torch.distributed.init_process_group('nccl', device_id=dev)
    from digat_b200 import _lib
    _lib.require_device(local_rank)           # fails loudly without the sm_100a library / device

    if args.mode == 'train':
        rec = train_record(args, rank, local_rank, world, dev, steps=args.steps, cpu_baseline=not args.no_cpu_baseline)
        if rank == 0:
            print(json.dumps(rec))
    elif args.mode == 'train_tokens':
        if rank == 0:
            print(json.dumps(train_tokens_record(args, dev, steps=args.steps)))
    else:
        run_score(args, rank, local_rank, world, dev)
    if world > 1:
        torch.distributed.destroy_process_group()


def run_score(args, rank, local_rank, world, dev):
    from digat_b200 import _lib, scoring
    from digat_b200.graphEncoders import DIGAT

    cfg, sd, corpus = build_workload(args.workload, rank=rank, world=world)
    enc = DIGAT(cfg, D)
    enc.load_state_dict(sd)
    enc = enc.to(dev).eval()
    scorer = scoring.Scorer(enc, corpus, dev)
    scorer.cache_news_context()

    n_pairs = corpus.pair_behavior.shape[0]
    sharded = args.workload in SHARDED_WORKLOADS                 # this rank generated only its own behaviours
    lo, hi = (0, n_pairs) if sharded else scoring.shard_range(n_pairs, rank, world)   # contiguous shard of the ordered pair list
    total_steps = args.warmup + args.steps
    assert (hi - lo) >= total_steps * args.batch, 'shard too small for steps*batch'
    pair_beh = torch.from_numpy(corpus.pair_behavior[lo:hi]).to(dev)
    pair_news = torch.from_numpy(corpus.pair_news[lo:hi]).to(dev)
    n_batches = (hi - lo) // args.batch

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- resident path (value)
    def step_resident(s):
        a = s * args.batch
        return scorer.score_resident(pair_beh[a:a + args.batch], pair_news[a:a + args.batch])

    def index_batches(s0, s1):
        return ((pair_beh[(s % n_batches) * args.batch:(s % n_batches + 1) * args.batch],
                 pair_news[(s % n_batches) * args.batch:(s % n_batches + 1) * args.batch]) for s in range(s0, s1))

    # The clock sampler is started BEFORE the warm-up and must have delivered its first sample before the timed region
    # begins: its start-up (NVML initialisation) stalls kernel launches for tens of milliseconds, which used to land inside
    # the first timed steps every few runs (seen as 2-3x slower `value` at unchanged `e2e`).
    sampler = ClockSampler(local_rank)
    sampler.start()
    scoring.score_resident_batches(scorer, index_batches(0, args.warmup))
    t_wait = time.time()
    while not sampler.rows and sampler.mode != 'none' and time.time() - t_wait < 10.0:
        time.sleep(0.05)
    # A full (generation-2) garbage collection of a process that has imported torch walks ~10^6 objects: 50-150 ms during
    # which nothing is enqueued.  Every few runs one landed inside the timed steps (one step of 45-130 ms).  Collect now and
    # freeze the survivors so that collections inside the timed region only look at the objects created there.
    import gc
    gc.collect()
    gc.freeze()
    barrier()
    _lib.reset_launch_count()
    c_lo = sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    profile_range = os.environ.get('DIGAT_PROFILE_RANGE') == '1'     # `ncu --profile-from-start off`: exactly the timed steps
    if profile_range:
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    # the public pipelined driver: the flag kernels of batch k+1 are enqueued ahead of the encoder pass of batch k and
    # the host waits for their counts (the only synchronisation of a step) while that pass runs
    step_events = []
    outs = scoring.score_resident_batches(scorer, index_batches(args.warmup, total_steps), events=step_events)
    e1.record()
    if profile_range:
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
    barrier()
    launches = _lib.launch_count()
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'logits.npy' if world == 1 else 'logits_rank%d.npy' % rank),
                outs[-1].cpu().numpy())
    del outs
    ms_resident = _max_over_ranks(e0.elapsed_time(e1), world, dev)
    marks = [e0] + step_events
    step_ms = sorted(marks[k].elapsed_time(marks[k + 1]) for k in range(len(marks) - 1))
    scorer.check_index_errors()

    # ---------------------------------------------------------------- end-to-end path (host buffers)
    host = [scoring.host_batch(corpus, np.arange(lo + s * args.batch, lo + (s + 1) * args.batch), pin=True, config=cfg)
            for s in range(total_steps)]
    h2d = int(sum(t.numel() * t.element_size() for t in host[0]))
    res = torch.empty((total_steps, args.batch), dtype=torch.float32).pin_memory()
    scoring.score_host_batches(scorer, host[:args.warmup], res[:args.warmup])
    barrier()
    e0.record()
    # the public pipelined call: every timed step's H2D copy and D2H read is issued inside the timed region
    # (batch k+1's copies overlap batch k's kernels on a side stream)
    scoring.score_host_batches(scorer, host[args.warmup:total_steps], res[args.warmup:total_steps])
    e1.record()
    barrier()
    ms_e2e = _max_over_ranks(e0.elapsed_time(e1), world, dev)
    clocks = sampler.stats(c_lo, sampler.mark())
    del host

    # ---------------------------------------------------------------- sustained: >= --sustained seconds back to back
    sustained = None
    if args.sustained > 0:
        per_step = ms_resident / args.steps * 1e-3
        n_sus = max(args.steps, int(args.sustained / per_step * 1.05) + 1)          # same count on every rank
        if world > 1:
            t = torch.tensor([n_sus], device=dev, dtype=torch.int64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            n_sus = int(t.item())
        barrier()
        s_lo = sampler.mark()
        e0.record()
        scoring.score_resident_batches(scorer, index_batches(0, n_sus))
        e1.record()
        barrier()
        ms_sus = _max_over_ranks(e0.elapsed_time(e1), world, dev)
        sustained = {'value': world * n_sus * args.batch / (ms_sus * 1e-3), 'unit': 'pairs/s', 'seconds': ms_sus * 1e-3,
                     'steps': n_sus, 'ms_per_step': ms_sus / n_sus, 'clocks': sampler.stats(s_lo, sampler.mark()),
                     'note': 'the resident path back to back over this rank\'s shard (cyclically); same driver as `value`'}
    sampler.stop()

    # ---------------------------------------------------------------- per-kernel timing -> roofline (untimed pass)
    prof = _lib.start_profile()
    prof_preps = []
    for s in range(args.warmup, min(total_steps, args.warmup + 3)):
        a = s * args.batch
        prep = scorer.prepare_resident(pair_beh[a:a + args.batch], pair_news[a:a + args.batch])
        prof_preps.append(prep)
        scorer.score_prepared(prep)
    torch.cuda.synchronize()
    kernels = _lib.stop_profile()
    # what pruning keeps (for the layer kernel's efficiency figure): active user / news node rows per pair
    act_u = float(np.mean([p['prune'][1].shape[0] if p['prune'] is not None else args.batch * (cfg.max_history_num + cfg.category_num)
                           for p in prof_preps])) / args.batch
    act_n = float(np.mean([p['prune_n'][1].shape[0] if p['prune_n'] is not None else args.batch * cfg.news_graph_size
                           for p in prof_preps])) / args.batch

    pairs_total = world * args.steps * args.batch
    value = pairs_total / (ms_resident * 1e-3)
    e2e = pairs_total / (ms_e2e * 1e-3)

    train = None
    if not args.no_train and args.workload not in SHARDED_WORKLOADS:
        del scorer, pair_beh, pair_news
        torch.cuda.empty_cache()
        train = train_record(args, rank, local_rank, world, dev, steps=args.train_steps,
                             cpu_baseline=not args.no_cpu_baseline)

    if rank == 0:
        hbm_peak, tensor_peak, peak_src = _peaks()
        n_n, n_u, L = cfg.news_graph_size, cfg.max_history_num + cfg.category_num, cfg.graph_depth
        b_alg = algorithmic_bytes_per_pair(n_n, n_u, L)
        table = summarize_kernels(kernels, hbm_peak, tensor_peak, active_rows={n_u: act_u, n_n: act_n})
        top = table[0] if table else None
        roofline = None
        if top:
            traffic, traffic_note = None, None
            for tj in ('r2_traffic.json', 'r1_traffic.json'):           # DRAM bytes per launch from the ncu --set full captures
                tj = os.path.join(ROOT, 'profiles', tj)
                if os.path.isfile(tj):
                    ent = json.load(open(tj)).get(top['kernel'])
                    if ent:
                        traffic, traffic_note = ent['bytes'], ent['launch'] + ' / ' + ent['capture']
                        break
            roofline = {'kernel': top['kernel'], 'bound': top['bound'], 'achieved': top['achieved'], 'peak': top['peak'],
                        'unit': top['unit'], 'frac': top['achieved'] / top['peak'], 'traffic': traffic,
                        'traffic_note': traffic_note,
                        'share_of_step': top['share'], 'peak_source': peak_src, 'avg_launch_ms': top['avg_ms']}
        per_gpu = value / world                                   # one GPU's pairs/s against one GPU's HBM peak
        line = {
            'metric': 'impressions_scored_per_sec', 'value': value, 'unit': 'pairs/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_resident / args.steps,
            'step_ms': {'min': step_ms[0], 'median': step_ms[len(step_ms) // 2], 'max': step_ms[-1]},
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': args.workload, 'pairs_per_step_per_gpu': args.batch, 'SAG_neighbors': cfg.SAG_neighbors,
                       'SAG_hops': cfg.SAG_hops, 'news_graph_size': n_n, 'user_graph_size': n_u, 'graph_depth': L,
                       'D': D, 'n_news': int(corpus.news_embeddings.shape[0]),
                       'n_pairs': int(n_pairs) if not sharded else None,
                       'parallelism': 'pair-sharded x%d, no communication' % world,
                       'l2_policy': 'inputs larger than L2 (per-step intermediates ~%.1f GB)' %
                                    (args.batch * n_u * 3 * D * 4 / 1e9)},
            'e2e': {'value': e2e, 'unit': 'pairs/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': args.batch * 4,
                    'ms_per_step': ms_e2e / args.steps},
            'gpu_launches': launches,
            'clocks': clocks,
            'roofline': roofline,
            'roofline_path': {'bound': 'hbm', 'bytes_per_pair_alg': b_alg, 'achieved': per_gpu * b_alg / 1e9,
                              'peak': hbm_peak, 'unit': 'GB/s', 'frac': per_gpu * b_alg / 1e9 / hbm_peak, 'per': 'GPU',
                              'note': 'SURVEY 8(d) B_alg per pair x ONE GPU\'s pairs/s over one GPU\'s measured HBM peak; '
                                      'the path is tensor/ALU-bound, see DESIGN.md'},
            'sustained': sustained,
            'kernels': table[:10],
            'active_rows_per_pair': {'user_graph': act_u, 'news_graph': act_n, 'dense': {'user_graph': n_u, 'news_graph': n_n}},
        }
        if sharded:
            line['config']['scale'] = ('1.0 of BASELINE configs[4]: %d news, %d behaviours over %d ranks (%d on this rank, '
                                       '%d pairs)' % (WORKLOADS[args.workload][3], WORKLOADS[args.workload][4], world,
                                                      corpus.history.shape[0], n_pairs))
        if not args.no_cpu_baseline and world == 1:
            pps, sec, cores, n = oracle_pairs_per_second(cfg, sd, corpus, 64, args.cpu_budget)
            line['cpu_baseline'] = {'value': pps, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                                    'sample': '%d calls x 64 pairs of the same workload (%.1f s of CPU work), '
                                              'oracle/digat_oracle.py inference, torch CPU fp32' % (n, n * sec)}
        if train is not None:
            line['train'] = train
        print(json.dumps(line))


# -------------------------------------------------------------------------------------------------- training record
ORDER = ('news_graph_embeddings', 'news_graph', 'news_graph_mask', 'user_news_embedding', 'user_graph',
         'user_category_mask', 'user_category_indices')


def oracle_train_samples_per_second(cfg, sd, corpus, behaviours, news_num, budget_s):
    """CPU baseline of a training step: fwd + bwd of the oracle port through torch autograd (all host cores), on
    `behaviours` x `news_num` encoder rows (the Eq. (8) tensor autograd saves is 7.4 MB per row and layer)."""
    from digat_b200 import synth
    from oracle import digat_oracle as O
    import torch.nn.functional as F
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = {k: v.clone().requires_grad_(True) for k, v in O.cast_params(sd).items()}
    rows = behaviours * news_num
    batch = synth.make_batch(corpus, np.arange(rows))
    args = [batch[k] for k in ORDER]

    def step():
        for v in P.values():
            v.grad = None
        cn, cu = O.forward(P, *args)
        logits = O.logits(cn, cu).view(behaviours, news_num)
        (-F.log_softmax(logits, dim=1).select(1, 0)).mean().backward()
    step()
    n, t0 = 0, time.perf_counter()
    while True:
        step()
        n += 1
        el = time.perf_counter() - t0
        if el >= budget_s:
            break
    return n * behaviours / el, el / n, cores, n, rows


def ddp_gradient_check(dev, rank, world):
    """What tests/ddp_worker.py computes: gradients after DDP's NCCL all-reduce over `world` ranks (8 rows each) against
    single-process gradients on the union batch, max relative difference over all parameters (rank 0's view)."""
    from torch.nn.parallel import DistributedDataParallel as DDP
    from digat_b200 import synth
    from digat_b200.graphEncoders import DIGAT
    cfg = synth.make_config(graph_depth=2, dropout_rate=0.0)
    sd = synth.make_state_dict(cfg, seed=6)
    corpus = synth.make_corpus(cfg, n_news=300, n_behaviors=8 * world, mean_candidates=3.0, seed=3)
    batch = synth.make_batch(corpus, np.arange(8 * world))
    m = DIGAT(cfg, D)
    m.load_state_dict(sd)
    m = m.to(dev).train()
    ddp = DDP(m, device_ids=[dev.index])
    b = [batch[k][rank * 8:(rank + 1) * 8].to(dev) for k in ORDER]
    cn, cu = ddp(*b)
    (cn * cu).sum(1).mean().backward()
    torch.cuda.synchronize()
    worst = 0.0
    if rank == 0:
        m1 = DIGAT(cfg, D)
        m1.load_state_dict(sd)
        m1 = m1.to(dev).train()
        cn, cu = m1(*[batch[k].to(dev) for k in ORDER])
        (cn * cu).sum(1).mean().backward()
        torch.cuda.synchronize()
        g = dict(m.named_parameters())
        for k, v in m1.named_parameters():
            a, r = g[k].grad.double(), v.grad.double()
            worst = max(worst, float((a - r).abs().max() / r.abs().max().clamp_min(1e-30)))
    torch.distributed.barrier()
    return worst


def train_record(args, rank, local_rank, world, dev, steps, cpu_baseline=True):
    """BASELINE.json configs[2]: DIGAT training fwd+bwd on synthetic MIND-shaped batches, per-GPU batch = 64 behaviours
    x (1 + 4 negatives) = 320 rows (reference config.py:31,34), dropout 0.2, DDP gradient all-reduce over NCCL when
    launched with N>1 ranks, clip-norm 1 + Adam step as reference trainer.py:98-105.  News-encoder excluded (SURVEY 8d)."""
    import torch.nn.functional as F
    from digat_b200 import _lib, synth
    from digat_b200.model import Model
    workload = args.workload if args.workload not in SHARDED_WORKLOADS else 'mind_small_dev_n3_L3'
    N, hops, L = WORKLOADS[workload][:3]
    cfg = synth.make_config(SAG_neighbors=N, SAG_hops=hops, graph_depth=L, dropout_rate=0.2)
    sd = synth.make_state_dict(cfg, D=D, seed=0)
    corpus = synth.make_corpus(cfg, D=D, n_news=20000, n_behaviors=4096, mean_candidates=8.0, seed=rank)
    model = Model(cfg, D)
    model.graph_encoder.load_state_dict(sd)
    model = model.to(dev).train()
    # Gradient exchange: by default ONE all-reduce (mean) of the flat gradient buffer (digat_b200/training.py::FlatGradients)
    # inside the step, which -- unlike DDP's reducer hooks -- captures into the whole-step CUDA graph; --eager-train runs the
    # reference's arrangement instead (torch DistributedDataParallel around the model, trainer.py:19, eager).
    from digat_b200.training import FlatAdam, GraphedTrainStep, broadcast_parameters
    use_ddp = world > 1 and args.eager_train
    graphed = not args.eager_train
    # optimizer: the flat clip + Adam kernels (digat_b200/training.py::FlatAdam); the DDP arm keeps torch.optim.Adam
    opt = torch.optim.Adam(model.parameters(), lr=1e-4) if use_ddp else None
    bs, news_num = 64, 5
    warmup = max(args.warmup, 3)
    rng = np.random.Generator(np.random.PCG64(rank))
    emb = torch.from_numpy(corpus.news_embeddings).to(dev)
    node = torch.from_numpy(corpus.news_node_ID.astype(np.int64)).to(dev)
    ng, nm = torch.from_numpy(corpus.news_graph).to(dev), torch.from_numpy(corpus.news_graph_mask).to(dev)
    hist = torch.from_numpy(corpus.history.astype(np.int64)).to(dev)
    ug, cm, ci = (torch.from_numpy(x).to(dev) for x in (corpus.user_graph, corpus.user_category_mask, corpus.user_category_indices))

    def make_step_inputs():
        beh = torch.from_numpy(rng.integers(0, hist.shape[0], size=bs)).to(dev)
        cand = torch.from_numpy(rng.integers(1, emb.shape[0], size=(bs, news_num))).to(dev)
        return (emb[hist[beh]], ug[beh], cm[beh], ci[beh], emb[node[cand]], ng[cand], nm[cand])

    if use_ddp:
        # DDP hooks fire on the wrapped module's forward: route forward_embeddings through it
        class _Fwd(torch.nn.Module):
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, *a):
                return self.m.forward_embeddings(*a)
        fwd = torch.nn.parallel.DistributedDataParallel(_Fwd(model), device_ids=[local_rank])
        flat = None
    else:
        fwd = model.forward_embeddings
        broadcast_parameters(model)
        flat = FlatAdam(model.parameters(), lr=1e-4, max_norm=1.0, modules=(model,))

    def eager_step(inp):
        logits = fwd(*inp)
        loss = (-F.log_softmax(logits, dim=1).select(1, 0)).mean()
        if flat is None:
            opt.zero_grad(set_to_none=True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
        else:
            flat.zero_grad()
            loss.backward()
            flat.all_reduce_mean()                                # NCCL all-reduce over NVLink (no-op on one GPU)
            flat.step()                                           # clip_grad_norm 1 + Adam, two launches
        return loss

    inputs = [make_step_inputs() for _ in range(warmup + steps)]
    step = eager_step
    capture_note = None
    if graphed:
        try:
            gstep = GraphedTrainStep(lambda *a: eager_step(a), inputs[0], modules=(model,), distributed=world > 1)
            step = lambda inp: gstep(*inp)                      # noqa: E731
        except Exception as exc:                                # capture refused (e.g. NCCL inside the graph): stay eager
            graphed = False
            capture_note = 'graph capture failed, ran eagerly: %s' % str(exc).splitlines()[0][:200]
            torch.cuda.synchronize()
    for s_ in range(warmup):
        step(inputs[s_])
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s_ in range(warmup, warmup + steps):
        loss = step(inputs[s_])
    e1.record()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ms = _max_over_ranks(e0.elapsed_time(e1), world, dev)
    launches_timed = _lib.launch_count()
    final_loss = float(loss)

    # per-kernel table: one eager step through the profiling hooks (CUDA events around every C-ABI call)
    _lib.start_profile()
    e0.record()
    eager_step(inputs[warmup])
    e1.record()
    torch.cuda.synchronize()
    recs = _lib.stop_profile()
    eager_ms = e0.elapsed_time(e1)
    agg = {}
    for name, a, t in recs:
        e = agg.setdefault(name, [0.0, 0])
        e[0] += t
        e[1] += 1
    ours_ms = sum(v[0] for v in agg.values()) or 1.0
    kernels = [{'kernel': k, 'ms_per_step': v[0], 'launches': v[1], 'share_of_our_kernels': v[0] / ours_ms}
               for k, v in sorted(agg.items(), key=lambda kv: -kv[1][0])][:12]

    grad_check = ddp_gradient_check(dev, rank, world) if world > 1 else None
    rec = None
    if rank == 0:
        n_params = sum(p.numel() for p in model.parameters())
        rec = {'metric': 'train_samples_per_sec', 'value': world * steps * bs / (ms * 1e-3), 'unit': 'samples/s',
               'n_gpus': world, 'steps': steps, 'warmup': warmup, 'ms_per_step': ms / steps,
               'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
               'config': {'workload': workload + ':train', 'behaviours_per_gpu': bs, 'candidates': news_num,
                          'rows_per_gpu': bs * news_num, 'dropout': 0.2, 'optimizer': 'Adam + clip_grad_norm 1' + (' (torch.optim)' if use_ddp else ' (flat buffers, 2 kernel launches)'),
                          'execution': ('whole step (incl. the gradient all-reduce) replayed as one CUDA graph' if graphed
                                        else 'eager') + ('; ' + capture_note if capture_note else ''),
                          'parallelism': ('data parallel x%d, %s, %.1f MB fp32 per step' % (
                              world, 'torch DistributedDataParallel (bucketed NCCL all-reduce)' if use_ddp
                              else 'one NCCL all-reduce (mean) of the flat gradient buffer', n_params * 4 / 1e6))
                                         if world > 1 else 'single GPU (no collective)'},
               'gpu_launches': launches_timed if not graphed else sum(v[1] for v in agg.values()) * steps,
               'gpu_launches_note': 'C-ABI kernel launches (replayed from the captured graph)' if graphed else 'C-ABI kernel launches',
               'final_loss': final_loss,
               'eager_step_ms': eager_ms, 'our_kernels_ms_per_step': ours_ms, 'kernels': kernels}
        if grad_check is not None:
            rec['ddp_vs_single_process_grad_rel_diff'] = grad_check
        if cpu_baseline and world == 1:
            sps, sec, cores, n, rows = oracle_train_samples_per_second(cfg, sd, corpus, 12, news_num, min(args.cpu_budget, 10.0))
            rec['cpu_baseline'] = {'value': sps, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                                   'sample': '%d fwd+bwd steps of %d behaviours x %d candidates = %d encoder rows (%.1f s of CPU '
                                             'work), oracle/digat_oracle.py under torch autograd, CPU fp32' % (n, 12, news_num, rows, n * sec)}
    return rec


def train_tokens_record(args, dev, steps):
    """End-to-end training step of the reference from TOKEN tensors (model.py:54-77, trainer.py:86-105): MSA news encoder over the
    64 x 50 history titles and the 320 x n_n candidate-graph titles of a step, then the graph encoder, loss, backward through both,
    clip + Adam (FlatAdam).  Not part of BASELINE's metric (SURVEY 8(d) excludes the news encoder): an extra record.  Eager (the
    news encoder's training path reads an error flag on the host), one GPU."""
    import torch.nn.functional as F
    from digat_b200 import _lib, synth
    from digat_b200.model import Model
    from digat_b200.training import FlatAdam
    workload = args.workload if args.workload not in SHARDED_WORKLOADS else 'mind_small_dev_n3_L3'
    N, hops, L = WORKLOADS[workload][:3]
    cfg = synth.make_text_config(vocabulary_size=40000, SAG_neighbors=N, SAG_hops=hops, graph_depth=L, dropout_rate=0.2)
    model = Model(cfg)
    model.graph_encoder.load_state_dict(synth.make_state_dict(cfg, D=D, seed=0))
    model.news_encoder.load_state_dict(synth.make_msa_state_dict(cfg, seed=1))
    model = model.to(dev).train()
    corpus = synth.make_corpus(cfg, D=D, n_news=20000, n_behaviors=4096, mean_candidates=8.0, seed=0)
    tok, mask = synth.make_titles(cfg, 20000, seed=2)
    tok, mask = tok.to(dev), mask.to(dev)
    flat = FlatAdam(model.parameters(), lr=1e-4, max_norm=1.0, modules=(model,))
    bs, news_num = 64, 5
    rng = np.random.Generator(np.random.PCG64(0))
    node = torch.from_numpy(corpus.news_node_ID.astype(np.int64)).to(dev)
    ng, nm = torch.from_numpy(corpus.news_graph).to(dev), torch.from_numpy(corpus.news_graph_mask).to(dev)
    hist = torch.from_numpy(corpus.history.astype(np.int64)).to(dev)
    ug, cm, ci = (torch.from_numpy(x).to(dev) for x in (corpus.user_graph, corpus.user_category_mask, corpus.user_category_indices))

    def inputs():
        beh = torch.from_numpy(rng.integers(0, hist.shape[0], size=bs)).to(dev)
        cand = torch.from_numpy(rng.integers(1, tok.shape[0], size=(bs, news_num))).to(dev)
        return (tok[hist[beh]], mask[hist[beh]], ug[beh], cm[beh], ci[beh], tok[node[cand]], mask[node[cand]], ng[cand], nm[cand])

    def step(inp):
        logits = model(*inp)
        loss = (-F.log_softmax(logits, dim=1).select(1, 0)).mean()
        flat.zero_grad()
        loss.backward()
        flat.step()
        return loss
    warmup = max(args.warmup, 3)
    batches = [inputs() for _ in range(warmup + steps)]
    for i in range(warmup):
        step(batches[i])
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(warmup, warmup + steps):
        loss = step(batches[i])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    titles = bs * cfg.max_history_num + bs * news_num * cfg.news_graph_size
    return {'metric': 'train_samples_per_sec_from_tokens', 'value': steps * bs / (ms * 1e-3), 'unit': 'samples/s', 'n_gpus': 1,
            'steps': steps, 'warmup': warmup, 'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': workload + ':train_tokens', 'behaviours_per_gpu': bs, 'candidates': news_num,
                       'titles_per_step': titles, 'tokens_per_title': cfg.max_title_length, 'vocabulary': cfg.vocabulary_size,
                       'news_encoder': 'MSA 16 x 25, word_embedding_dim 300', 'dropout': 0.2,
                       'optimizer': 'Adam + clip_grad_norm 1 (flat buffers)', 'execution': 'eager'},
            'gpu_launches': _lib.launch_count(), 'final_loss': float(loss)}


def summarize_kernels(records, hbm_peak, tensor_peak, active_rows=None):
    """records: [(name, args, ms)] from _lib.stop_profile -> per-kernel-class share and roofline numbers.
    active_rows {n: mean node rows per graph that survive pruning}: the fused layer kernel gets a second figure,
    `needed` = the bytes the PRUNED result needs (5 rows-worth of D floats per active node + the adjacency), next to the
    dense-layout figure `achieved` (every node row counted, as SURVEY 8(d) defines B_alg)."""
    agg = {}
    for name, a, ms in records:
        work2 = None
        if name == 'digat_graph_layer_fwd':
            B, n, Dd = a[6], a[7], a[8]
            key = '%s[n=%d]' % (name, n)
            work, bound = B * (5 * n * Dd * 4 + n * n + Dd * 4), 'hbm'
            if a[19] and active_rows and n in active_rows:              # row_active given: pruned evaluation
                work2 = B * (5 * active_rows[n] * Dd * 4 + n * n + Dd * 4)
        elif name == 'digat_linear_f32' or name == 'digat_linear_tf32x3':
            M, N, K = (a[7], a[8], a[9]) if name == 'digat_linear_f32' else (a[8], a[9], a[10])
            key = '%s[N=%d,K=%d,%s]' % (name, N, K, 'M>2048' if M > 2048 else 'M<=2048')
            work, bound = 2.0 * M * N * K, 'tensor'
        elif name == 'digat_attention_pool_fwd':
            B, m, Dd = a[12], a[13], a[14]
            key = '%s[m=%d]' % (name, m)
            work, bound = B * (m * Dd * 4 * (2 if a[3] else 1) + 2 * Dd * 4), 'hbm'
        elif name == 'digat_topic_segment_fwd':
            B, H, S, Dd = a[12], a[13], a[14], a[15]
            key, work, bound = name, B * (H * Dd * 4 + S * Dd * 4 + Dd * 4 + H * 8), 'hbm'
        elif name in ('digat_gather_sag_i32',):
            key, work, bound = name, a[6] * a[3] * a[7] * 4 * 2, 'hbm'
        elif name == 'digat_gather_rows_i32':
            key, work, bound = name, a[5] * a[6] * 4 * 2, 'hbm'
        elif name == 'digat_build_user_nodes':
            key, work, bound = name, a[6] * (a[7] + a[8]) * a[9] * 4 * 2, 'hbm'
        else:
            key, work, bound = name, 0.0, 'hbm'
        e = agg.setdefault(key, {'kernel': key, 'bound': bound, 'ms': 0.0, 'work': 0.0, 'work2': 0.0, 'launches': 0})
        e['ms'] += ms
        e['work'] += work
        e['work2'] += work2 if work2 is not None else work
        e['launches'] += 1
    total = sum(e['ms'] for e in agg.values()) or 1.0
    out = []
    for e in agg.values():
        if e['bound'] == 'hbm':
            ach, peak, unit = e['work'] / (e['ms'] * 1e-3) / 1e9, hbm_peak, 'GB/s'
        else:
            ach, peak, unit = e['work'] / (e['ms'] * 1e-3) / 1e12, tensor_peak, 'TFLOP/s'
        row = {'kernel': e['kernel'], 'bound': e['bound'], 'share': e['ms'] / total, 'avg_ms': e['ms'] / e['launches'],
               'launches': e['launches'], 'achieved': ach, 'peak': peak, 'unit': unit, 'frac': ach / peak}
        if e['work2'] != e['work']:
            need = e['work2'] / (e['ms'] * 1e-3) / 1e9
            row.update(needed_GBps=need, frac_needed=need / peak,
                       note='achieved = dense-layout bytes; needed = bytes of the pruned result (active rows only)')
        out.append(row)
    out.sort(key=lambda r: -r['share'])
    return out


if __name__ == '__main__':
    main()
