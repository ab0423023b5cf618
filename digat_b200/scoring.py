"""Scoring driver over the sm_100a graph encoders (DIGAT and the five ablations): the device-side part of reference
util.compute_scores (util.py:34-69) -- SAG neighbour gather, the cached per-news context (c_n0; util.py:39-50 dispatches
it per encoder), and the per-batch gathers + Model.inference -- with every gather done by the kernels of libdigat_sm100.so.
The encoder owns its scoring schedule (``_encode``), what is cached per news (``_news_cache``) and which news-side nodes
it reads per pair (``SCORE_NEWS_NODES``).

Two ways in:
* ``score_host_batch``  takes the HOST tensors the reference DataLoader yields (util.py:56: user_title_index,
  user_graph, user_category_mask, user_category_indices, news_ID, news_graph, news_graph_mask), copies them to the
  device and scores them; ``score_host_batches`` does it for a whole DataLoader, pipelined (the end-to-end "e2e" path
  of bench.py);
* ``score_resident``    takes only (behaviour index, news id) per pair; graphs, masks and tables stay resident in HBM;
  ``score_resident_batches`` / ``evaluate_resident`` are its pipelined drivers (scores, on-GPU ranks and metrics).
A batch is prepared in two halves (``begin_*``: launches only; ``finish_prepare``: one event wait for four list lengths)
so that the drivers can enqueue batch k+1's first half ahead of batch k's encoder pass (see ``_pipelined``).
Pairs are independent, so multi-GPU inference shards the pair list with no communication (``shard_range``).
"""
import math

import numpy as np
import torch

from . import _lib
from .model import logits


def shard_range(n_items: int, rank: int, world_size: int):
    """Contiguous shard [lo, hi) of an ordered pair list (scores are concatenated in rank order afterwards)."""
    per = (n_items + world_size - 1) // world_size
    lo = min(rank * per, n_items)
    return lo, min(lo + per, n_items)


class Scorer:
    def __init__(self, encoder, corpus, device, build_user_graphs_on_device=False):
        """encoder: one of the six graph encoders (DIGAT and the five ablations of ablation_encoders.ENCODERS) on `device`;
        the scores are that encoder's ``inference``.  corpus: digat_b200.synth.Corpus (host numpy).

        build_user_graphs_on_device: derive user_graph / category mask / segment ids from the [N_beh,H] category table
        with the CUDA builder (graphs.build_user_graphs_device; bit-identical to MIND_corpus.py:143-176) instead of
        uploading the [N_beh,n_u,n_u] bool array (4.6 KB per behaviour vs 200 B)."""
        from .ablation_encoders import ENCODERS
        schedule = next((c for c in type(encoder).__mro__ if '_encode' in vars(c)), None)   # whose _encode would run
        if schedule not in ENCODERS.values():
            raise RuntimeError('Scorer: no scoring schedule for %s; supported encoders: %s'
                               % (type(encoder).__name__, ', '.join(c.__name__ for c in ENCODERS.values())))
        self.enc = encoder.eval()
        self.dev = torch.device(device)
        if self.dev.type == 'cuda' and self.dev.index is not None and self.dev.index != torch.cuda.current_device():
            raise RuntimeError('Scorer(device=%s): kernels launch on the current device (cuda:%d) -- call '
                               'torch.cuda.set_device first' % (self.dev, torch.cuda.current_device()))
        _lib.require_device(self.dev.index if self.dev.index is not None else torch.cuda.current_device())
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        self.table = t(corpus.news_embeddings)                  # [N,D]   cached news representations (util.py:20-33)
        self.node_id = t(corpus.news_node_ID)                   # [N,n_n] int32 (util.py:34)
        self.news_graph = t(corpus.news_graph)                  # [N,n_n,n_n] bool
        self.news_mask = t(corpus.news_graph_mask)              # [N,n_n] bool (util.py:35)
        self.history = t(corpus.history)                        # [Nb,H] int32
        if build_user_graphs_on_device or corpus.user_graph is None:
            from . import graphs
            H = corpus.history.shape[1]
            C = encoder.category_num - 1 if hasattr(encoder, 'category_num') else corpus.user_category_mask.shape[1] - 1
            cat = t(corpus.history_category)
            self.user_graph, self.cmask, self.cidx = graphs.build_user_graphs_device(cat, (cat < C).sum(dim=1), H, C)
        else:
            self.user_graph = t(corpus.user_graph)              # [Nb,nu,nu] bool
            self.cmask = t(corpus.user_category_mask)
            self.cidx = t(corpus.user_category_indices)
        self.n_news, self.D = self.table.shape
        self.n_n = self.node_id.shape[1]
        self.err = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.c_n0 = None                                        # the encoder's per-news cache (_news_cache), or None
        self._c_n0_weights = None                               # the packed-weight generation c_n0 was computed with
        self._first_node = None                                 # [N] int32 node_id[:, 0] (SCORE_NEWS_NODES = 'first')

    def _st(self):
        return torch.cuda.current_stream().cuda_stream

    def gather_sag(self, news_idx):
        """[B] int32 news ids -> [B, n_n, D] SAG node embeddings (util.py:35-36 + :66 without the [N,n_n,D] cache)."""
        B = news_idx.shape[0]
        out = torch.empty((B, self.n_n, self.D), device=self.dev, dtype=torch.float32)
        _lib.call('digat_gather_sag_i32', self.table.data_ptr(), self.n_news, self.node_id.data_ptr(), self.n_n,
                  news_idx.data_ptr(), out.data_ptr(), B, self.D, self.err.data_ptr(), self._st())
        return out

    def gather_rows(self, table, idx):
        """out[r] = table[idx[r]] for a contiguous table [N, ...] (a row is all trailing dimensions)."""
        rows = idx.numel()
        width = math.prod(table.shape[1:])
        out = torch.empty((rows,) + tuple(table.shape[1:]), device=self.dev, dtype=torch.float32)
        _lib.call('digat_gather_rows_i32', table.data_ptr(), table.shape[0], idx.data_ptr(), out.data_ptr(),
                  width, rows, width, self.err.data_ptr(), self._st())
        return out

    def news_nodes(self, news_idx):
        """The news-side node embeddings the encoder's scoring schedule reads per pair (its SCORE_NEWS_NODES): the SAG
        [B,n_n,D], the candidate's own embedding [B,1,D] (SAG node 0) or None."""
        kind = self.enc.SCORE_NEWS_NODES
        if kind == 'graph':
            return self.gather_sag(news_idx)
        if kind == 'first':
            if self._first_node is None:
                self._first_node = self.node_id[:, 0].contiguous()
            return self.gather_rows(self.table, self._first_node.index_select(0, news_idx.long())).view(-1, 1, self.D)
        if kind == 'none':
            return None
        raise RuntimeError('%s.SCORE_NEWS_NODES must be graph, first or none (got %r)' % (type(self.enc).__name__, kind))

    def user_nodes(self, hist_idx):
        """[B,H] int32 history ids -> X_u [B, H+C, D] = [gathered history ; topic nodes] (util.py:65 + graphEncoders.py:191)."""
        w = self.enc._weights()
        B, H = hist_idx.shape
        C = w['topic'].shape[0]
        Xu = torch.empty((B, H + C, self.D), device=self.dev, dtype=torch.float32)
        _lib.call('digat_build_user_nodes', self.table.data_ptr(), self.n_news, hist_idx.data_ptr(), 0,
                  w['topic'].data_ptr(), Xu.data_ptr(), B, H, C, self.D, self.err.data_ptr(), self._st())
        return Xu

    def cache_news_context(self, batch_size=1024):
        """The encoder's per-news cache (_news_cache) for every news, in chunks of batch_size news: c_n0 (util.py:37-44)
        for DIGAT, Seq_SA (its sequence context) and User_graph_wo_inter; c_n^(0..L) [N, L+1, D] for the encoders with a
        vanilla-GAT news graph; None for wo_SA."""
        w = self.enc._weights()
        c = None
        with torch.no_grad():
            for lo in range(0, self.n_news, batch_size):
                hi = min(lo + batch_size, self.n_news)
                ids = torch.arange(lo, hi, device=self.dev, dtype=torch.int32)
                part = self.enc._news_cache(w, self.gather_sag(ids), self.news_graph[lo:hi], self.news_mask[lo:hi])
                if part is None:
                    break
                if c is None:
                    c = torch.empty((self.n_news,) + tuple(part.shape[1:]), device=self.dev, dtype=torch.float32)
                c[lo:hi] = part
        self.c_n0, self._c_n0_weights = c, w
        return c

    # ------------------------------------------------------------------------------------------------------------
    # A batch is scored in two steps.  prepare_* does everything that needs the HOST to look at device data (the
    # impression boundaries and the pruning lists are nonzero() calls, i.e. stream synchronisations) and depends on the
    # batch's integer/bool inputs only; score_prepared then launches the encoder without a single synchronisation.
    # score_host_batches runs prepare for batch k+1 on a side stream while batch k is encoded.
    def begin_resident(self, beh_idx, news_idx, share_user_graphs=True):
        """First half of a batch's preparation: launches only.  beh_idx, news_idx: [B] device tensors (any integer
        dtype); everything else is already in HBM."""
        enc = self.enc
        with torch.no_grad():
            nl, bl = news_idx.long(), beh_idx.long()
            prep = dict(news=news_idx.to(torch.int32), An=self.news_graph.index_select(0, nl),
                        Mn=self.news_mask.index_select(0, nl), Mc=self.cmask.index_select(0, bl), share=None)
            first = None
            if share_user_graphs and bl.shape[0] >= 2:
                first = torch.ones(bl.shape[0], dtype=torch.bool, device=bl.device)
                first[1:] = bl[1:] != bl[:-1]                            # impression boundaries in the ordered pair list
                prep['share'] = (torch.cumsum(first, 0) - 1).to(torch.int32)
            # flags straight from the resident per-behaviour tables (read through the behaviour index)
            uf = enc._user_flags(self.user_graph, prep['Mc'], self.cidx, bl.to(torch.int32))
            nf, sf = enc._news_flags(prep['An'], prep['Mn']), enc._segment_flags(prep['Mc'])
            state = enc.compact_begin([first, None if uf is None else uf[0], nf, sf])
        return dict(kind='resident', prep=prep, bl=bl, first=first, uf=uf, nf=nf, sf=sf, state=state)

    def begin_device_batch(self, user_title_index, user_graph, user_category_mask, user_category_indices, news_ID,
                           news_graph, news_graph_mask, share_user_graphs=True):
        """The same for the 7 tensors of one reference DataLoader batch (util.py:56), already on the device.

        The DataLoader repeats the user tensors for every candidate of an impression (MIND_dataset.py:97-102).
        Consecutive rows with the same clicked-news history have the same user graph / category tensors (they are
        functions of the history, MIND_corpus.py:143-176), so they are detected here and encoded through the
        shared-user-graph path (bit-identical results)."""
        enc = self.enc
        with torch.no_grad():
            hist = user_title_index.to(torch.int32)
            prep = dict(news=news_ID.to(torch.int32), An=news_graph, Mn=news_graph_mask, Mc=user_category_mask, share=None,
                        hist=hist, Au=user_graph, ci=user_category_indices)
            first = None
            if share_user_graphs and hist.shape[0] >= 2:
                first = torch.ones(hist.shape[0], dtype=torch.bool, device=hist.device)
                first[1:] = (hist[1:] != hist[:-1]).any(dim=1)
                prep['share'] = (torch.cumsum(first, 0) - 1).to(torch.int32)
            uf = enc._user_flags(user_graph, user_category_mask, user_category_indices, None)     # per-pair graphs
            nf, sf = enc._news_flags(news_graph, news_graph_mask), enc._segment_flags(user_category_mask)
            state = enc.compact_begin([first, None if uf is None else uf[0], nf, sf])
        return dict(kind='device', prep=prep, first=first, uf=uf, nf=nf, sf=sf, state=state)

    def finish_prepare(self, begun):
        """Second half: ONE host wait (an event recorded right behind the flag kernels, so nothing enqueued after
        begin_* delays it) for the counts of the impression boundaries and of the three pruning lists; the rest is launches."""
        enc, prep = self.enc, begun['prep']
        with torch.no_grad():
            comp = enc.compact_finish(begun['state'], 4)
            prep['first_rows'] = None if begun['first'] is None else comp[0][0]   # first pair of every distinct behaviour
            if begun['kind'] == 'resident':
                bl = begun['bl']
                if begun['first'] is not None:
                    bl = bl.index_select(0, comp[0][0].long())           # one row per behaviour: node tables, graphs, segment ids
                prep.update(hist=self.history.index_select(0, bl), Au=self.user_graph.index_select(0, bl),
                            ci=self.cidx.index_select(0, bl))
            elif begun['first'] is not None:
                rows = comp[0][0].long()
                prep.update(hist=prep['hist'].index_select(0, rows), Au=prep['Au'].index_select(0, rows),
                            ci=prep['ci'].index_select(0, rows))
            prep['prune'], prep['prune_n'], prep['seg_prune'] = self._pack_lists(begun['uf'], begun['nf'], begun['sf'], comp[1:])
        return prep

    def prepare_resident(self, beh_idx, news_idx, share_user_graphs=True):
        return self.finish_prepare(self.begin_resident(beh_idx, news_idx, share_user_graphs))

    def prepare_device_batch(self, *device_tensors, share_user_graphs=True):
        return self.finish_prepare(self.begin_device_batch(*device_tensors, share_user_graphs=share_user_graphs))

    @staticmethod
    def _pack_lists(uf, nf, sf, comp):
        cu, cn, cs = comp
        prune = prune_n = seg_prune = None
        if cu is not None and cu[0].shape[0] < uf[0].numel():
            prune = (uf[0], cu[0], cu[1], uf[1])
        if cn is not None and cn[0].shape[0] < nf.numel():
            prune_n = (nf, cn[0], cn[1])
        if cs is not None and cs[0].shape[0] < sf.numel():
            seg_prune = cs
        return prune, prune_n, seg_prune

    def score_prepared(self, prep):
        """Gathers + encoder + logits of a prepared batch: kernel launches only, no host synchronisation."""
        w = self.enc._weights()
        if self._c_n0_weights is not w:                          # the reference recomputes it per compute_scores call
            self.cache_news_context()                            # (util.py:37-44); here: whenever the weights were repacked
        with torch.no_grad():
            Xn = self.news_nodes(prep['news'])
            Xu = self.user_nodes(prep['hist'])                           # one node tensor per behaviour when shared
            c0 = None if self.c_n0 is None else self.gather_rows(self.c_n0, prep['news'])   # the pairs' cache rows
            cn, cu = self.enc._encode(w, Xn, prep['An'], prep['Mn'], Xu, prep['Au'], prep['Mc'], prep['ci'], c0,
                                      share=prep['share'],
                                      lists=(prep['prune'], prep['prune_n'], prep['seg_prune']),
                                      first_rows=prep.get('first_rows'))
            return logits(cn, cu)

    def score_resident(self, beh_idx, news_idx, share_user_graphs=True):
        """beh_idx, news_idx: [B] device tensors (any integer dtype).  Everything else is already in HBM.

        share_user_graphs: the pairs of one impression are consecutive in the reference's pair list
        (MIND_corpus.py:295-297) and share the user graph.  Its node build, its layer-0 projection GEMM and its
        adjacency are then computed / read once per distinct behaviour and indexed per pair (bit-identical results:
        the same rows go through the same kernels; tests/test_gpu_scoring.py)."""
        return self.score_prepared(self.prepare_resident(beh_idx, news_idx, share_user_graphs))

    def score_host_batch(self, user_title_index, user_graph, user_category_mask, user_category_indices, news_ID,
                         news_graph, news_graph_mask, share_user_graphs=True):
        """The reference hot loop body (util.py:56-68) on HOST tensors (pinned for async copies)."""
        return self.score_device_batch(*self.stage_host_batch(user_title_index, user_graph, user_category_mask,
                                                              user_category_indices, news_ID, news_graph,
                                                              news_graph_mask), share_user_graphs=share_user_graphs)

    def stage_host_batch(self, *host_tensors):
        """Host -> device copies of one DataLoader batch on the CURRENT stream (asynchronous for pinned tensors)."""
        return tuple(x.to(self.dev, non_blocking=True) for x in host_tensors)

    def score_device_batch(self, *device_tensors, share_user_graphs=True):
        """score_host_batch after its copies: the same 7 tensors, already on the device."""
        return self.score_prepared(self.prepare_device_batch(*device_tensors, share_user_graphs=share_user_graphs))

    def check_index_errors(self):
        if int(self.err.item()) != 0:
            self.err.zero_()
            raise RuntimeError('index out of range in a gather (reference: index_select raises)')
        self.enc.check_index_errors()


def host_batch(corpus, pair_ids, pin=False, config=None):
    """The 7 host tensors the reference's MIND_DevTest_Dataset + DataLoader yield for these pairs (MIND_dataset.py:97-102).
    config: needed only for a corpus made without host user graphs (synth.make_corpus(build_user_graph=False))."""
    b = corpus.pair_behavior[pair_ids]
    nid = corpus.pair_news[pair_ids]
    if corpus.user_graph is None:
        from . import synth
        ub, inv = np.unique(b, return_inverse=True)
        g, cm, ci = synth.user_graphs_of(corpus, config, ub)
        ug, ucm, uci = g[inv], cm[inv], ci[inv]
    else:
        ug, ucm, uci = corpus.user_graph[b], corpus.user_category_mask[b], corpus.user_category_indices[b]
    out = (torch.from_numpy(corpus.history[b]), torch.from_numpy(ug),
           torch.from_numpy(ucm), torch.from_numpy(uci),
           torch.from_numpy(nid.astype(np.int64)), torch.from_numpy(corpus.news_graph[nid]),
           torch.from_numpy(corpus.news_graph_mask[nid]))
    if pin:
        out = tuple(x.pin_memory() for x in out)
    return out


def _pipelined(scorer: Scorer, items, begin, results, events=None):
    """Software pipelining on ONE compute stream.  In stream order:  ... flags(k+1) | encoder(k) | lists(k+1), flags(k+2)
    | encoder(k+1) ...  The host waits (once per batch) on an event recorded right behind flags(k+1), i.e. while the GPU is
    entering encoder(k); it then enqueues the list building of batch k+1 and the next round.  The GPU never waits for the
    host as long as a round's enqueue time (about 2 ms) is shorter than an encoder pass, and nothing depends on how the GPU
    schedules concurrent streams (a staging stream that ran concurrently was starved for up to 100 ms every few runs)."""
    main = torch.cuda.current_stream(scorer.dev)
    outs = []
    it = iter(items)
    nxt = next(it, None)
    prep = scorer.finish_prepare(begin(nxt)) if nxt is not None else None
    k = 0
    while prep is not None:
        nxt = next(it, None)
        begun = begin(nxt) if nxt is not None else None           # flags of batch k+1: ahead of encoder(k) in the stream
        scores = scorer.score_prepared(prep)                      # launches only
        if results is not None:
            results[k].copy_(scores, non_blocking=True)
        outs.append(scores)
        if events is not None:                                    # per-batch completion events (diagnostics)
            ev_done = torch.cuda.Event(enable_timing=True)
            ev_done.record(main)
            events.append(ev_done)
        prep = scorer.finish_prepare(begun) if begun is not None else None
        k += 1
    return outs


def score_host_batches(scorer: Scorer, host_batches, results=None, share_user_graphs=True):
    """The reference hot loop (util.py:56-69) over an iterable of HOST batches (7-tuples, ideally pinned), pipelined:
    the host->device copies of batch k+1 run on a copy stream and its index preparation is enqueued ahead of the encoder
    pass of batch k; the scores of batch k go back to ``results[k]`` (pinned host tensors, optional) asynchronously.
    Every batch's host->device copy and device->host read happens inside this call.  Returns the device score tensors."""
    main = torch.cuda.current_stream(scorer.dev)
    side = getattr(scorer, '_copy_stream', None)
    if side is None:
        side = scorer._copy_stream = torch.cuda.Stream(device=scorer.dev)

    def begin(hb):
        with torch.cuda.stream(side):                             # DMA copies only: they overlap the running encoder pass
            dev_t = scorer.stage_host_batch(*hb)
            ev = torch.cuda.Event()
            ev.record(side)
        for t in dev_t:
            t.record_stream(main)                                 # allocated on the copy stream, consumed on the main one
        main.wait_event(ev)
        return scorer.begin_device_batch(*dev_t, share_user_graphs=share_user_graphs)

    return _pipelined(scorer, host_batches, begin, results)


def score_resident_batches(scorer: Scorer, index_batches, results=None, share_user_graphs=True, events=None):
    """The same pipeline for the resident path: ``index_batches`` yields (behaviour index, news id) device tensors."""
    return _pipelined(scorer, index_batches,
                      lambda ib: scorer.begin_resident(ib[0], ib[1], share_user_graphs=share_user_graphs), results, events)


def compute_scores(scorer: Scorer, corpus, batch_size: int, rank: int = 0, world_size: int = 1):
    """Scores this rank's shard of the ordered pair list through the (pipelined) host-batch path; returns a numpy array."""
    lo, hi = shard_range(corpus.pair_behavior.shape[0], rank, world_size)
    batches = (host_batch(corpus, np.arange(s, min(s + batch_size, hi)), pin=True) for s in range(lo, hi, batch_size))
    outs = score_host_batches(scorer, batches)
    scorer.check_index_errors()
    if not outs:
        return np.zeros(0, dtype=np.float32)
    return torch.cat(outs).cpu().numpy()


def evaluate_resident(scorer: Scorer, corpus, batch_size: int = 4096, rank: int = 0, world_size: int = 1,
                      on_single_class='raise'):
    """Device-resident replacement of the reference's evaluation loop (util.compute_scores, util.py:51-80, followed by
    evaluate.scoring): pairs are (behaviour index, news id) only, graphs and tables stay in HBM, and the per-impression
    ranking and metrics run on the GPU (csrc/builders.cuh).  Shards whole impressions across ranks (no communication).

    Returns dict(scores [P_local] f32 tensor, ranks [P_local] i32 tensor, offsets, metrics (auc, mrr, ndcg5, ndcg10))."""
    from . import evaluate
    off_all = evaluate.impression_offsets(corpus.pair_behavior)
    n_imp = off_all.shape[0] - 1
    i_lo, i_hi = shard_range(n_imp, rank, world_size)
    lo, hi = int(off_all[i_lo]), int(off_all[i_hi])
    dev = scorer.dev
    beh = torch.from_numpy(corpus.pair_behavior[lo:hi]).to(dev)
    news = torch.from_numpy(corpus.pair_news[lo:hi]).to(dev)
    outs = score_resident_batches(scorer, ((beh[s:s + batch_size], news[s:s + batch_size])
                                           for s in range(0, hi - lo, batch_size)))
    scores = torch.cat(outs) if outs else torch.empty(0, device=dev, dtype=torch.float32)
    scorer.check_index_errors()
    off = torch.from_numpy(off_all[i_lo:i_hi + 1] - lo).to(dev)
    ranks = evaluate.rank_pairs_device(scores, off)
    m = evaluate.metrics_device(ranks, torch.from_numpy(corpus.labels[lo:hi]).to(dev), off, on_single_class)
    return dict(scores=scores, ranks=ranks, offsets=off, metrics=m)
