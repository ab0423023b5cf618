"""Prints the end-to-end error of the CUDA path vs the golden fp32 / fp64 reference vectors (run on the GPU box)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tests.helpers import CASES, case_inputs, load_golden, rel_err
from digat_b200.graphEncoders import DIGAT
from digat_b200.model import logits
for name in CASES:
    cfg, sd, corpus, batch = case_inputs(name)
    z, meta = load_golden(name)
    m = DIGAT(cfg, 400); m.load_state_dict(sd); m = m.cuda().eval()
    b = {k: v.cuda() for k, v in batch.items()}
    # replicate rows so that every GEMM takes the tensor-core path (M >= 256)
    rep = 64
    bb = {k: v.repeat(rep, *([1] * (v.dim() - 1))) for k, v in b.items()}
    args = (bb['news_graph_embeddings'], bb['news_graph'], bb['news_graph_mask'], bb['user_news_embedding'],
            bb['user_graph'], bb['user_category_mask'], bb['user_category_indices'])
    with torch.no_grad():
        fn, fu = m.forward(*args)
        lg = logits(fn, fu)
    B = batch['news_graph'].shape[0]
    lg = lg[:B].cpu().numpy()
    print(name, 'logits: vs ref32 %.2e  vs ref64 %.2e  (ref32 vs ref64 %.2e)  ctx vs ref32 %.2e %.2e' % (
        rel_err(lg, z['ref32_logits']), rel_err(lg, z['ref64_logits']), rel_err(z['ref32_logits'], z['ref64_logits']),
        rel_err(fn[:B].cpu().numpy(), z['ref32_fwd_news_ctx']), rel_err(fu[:B].cpu().numpy(), z['ref32_fwd_user_ctx'])))
