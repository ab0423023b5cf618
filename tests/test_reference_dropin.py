"""The "one import line" claim of INTEGRATION.md, executed: the UNMODIFIED reference ``model.py`` is imported with
``graphEncoders`` resolved to ``digat_b200.graphEncoders`` and driven through ``Model.__init__`` (string dispatch,
model.py:18-31), ``load_state_dict`` of a checkpoint written by the reference's own encoder (main.py:23,36) and the argument
plumbing of ``Model.inference`` / ``Model.forward`` (model.py:54-90).  The reference code is not part of this repository:
these tests run when DIGAT_REFERENCE_ROOT names a checkout of it and skip otherwise.  No kernel is launched -- the
numerical side of the same loop is tests/test_gpu_dropin.py."""
import importlib.util
import os
import sys
import types

import pytest
import torch

from oracle.ref_loader import REFERENCE_ROOT, load_reference, reference_available

pytestmark = pytest.mark.skipif(not reference_available(), reason='needs the original DIGAT code: set DIGAT_REFERENCE_ROOT')

ENCODERS = ['DIGAT', 'wo_SA', 'Seq_SA', 'wo_interaction', 'news_graph_wo_inter', 'user_graph_wo_inter']


def _import_reference_model_over_ours():
    """reference model.py with `import graphEncoders` bound to digat_b200.graphEncoders and a stub news encoder (the
    reference's NewsEncoder.__init__ opens a word-embedding pickle that only exists after its preprocessing)."""
    import digat_b200.graphEncoders as ours
    load_reference()                                        # installs the torchtext / sentence_transformers / scatter stubs
    stub = types.ModuleType('newsEncoders')

    class _News(torch.nn.Module):
        def __init__(self, config):
            super().__init__()
            self.news_embedding_dim = config.MSA_head_num * config.MSA_head_dim
            self.table = torch.nn.Embedding(config.vocabulary_size, self.news_embedding_dim)

        def initialize(self):
            pass

        def forward(self, title_text, title_mask):          # [B, news_num, T] -> [B, news_num, D]
            return self.table(title_text).mean(dim=2)
    stub.MSA = stub.CNN = _News
    saved = {k: sys.modules.get(k) for k in ('graphEncoders', 'newsEncoders', 'model')}
    sys.modules['graphEncoders'], sys.modules['newsEncoders'] = ours, stub
    try:
        spec = importlib.util.spec_from_file_location('reference_model_over_digat_b200', os.path.join(REFERENCE_ROOT, 'model.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod, ours


def _config(graph_encoder, L=2):
    from digat_b200 import synth
    return synth.make_config(graph_depth=L, graph_encoder=graph_encoder, MSA_head_num=16, MSA_head_dim=25,
                             vocabulary_size=50, max_title_length=8, word_embedding_dim=300)


@pytest.mark.parametrize('name', ENCODERS)
def test_reference_model_builds_over_our_encoders_and_loads_reference_checkpoints(name):
    ref_model, ours = _import_reference_model_over_ours()
    ge_ref = load_reference()[0]
    cfg = _config(name)
    model = ref_model.Model(cfg)                                              # the reference's own dispatch, model.py:18-31
    assert type(model.graph_encoder).__module__.startswith('digat_b200.')
    assert model.model_name == 'MSA-' + name
    cls = {'news_graph_wo_inter': 'News_graph_wo_inter', 'user_graph_wo_inter': 'User_graph_wo_inter'}.get(name, name)
    ref_enc = getattr(ge_ref, cls)(cfg, 400)
    ref_enc.initialize()
    ckpt = {'graph_encoder.' + k: v for k, v in ref_enc.state_dict().items()}
    ckpt.update({'news_encoder.' + k: v for k, v in model.news_encoder.state_dict().items()})
    model.load_state_dict(ckpt)                                               # strict: every key, every shape (main.py:23,36)
    assert [k for k, _ in model.graph_encoder.named_parameters()] == [k for k, _ in ref_enc.named_parameters()]
    model.initialize()                                                        # model.py:42-44
    assert model.graph_encoder.max_history_num == 50                          # util.py:19
    # trainer.py:25-28 groups parameters by the 'graph_encoder.' prefix
    assert all(k.startswith(('graph_encoder.', 'news_encoder.')) for k, _ in model.named_parameters())


def test_reference_model_inference_and_forward_hand_our_encoder_the_reference_argument_order():
    ref_model, ours = _import_reference_model_over_ours()
    cfg = _config('DIGAT')
    model = ref_model.Model(cfg)
    B, n_n, n_u, D, H, C1 = 6, cfg.news_graph_size, 68, 400, 50, 19
    seen = {}

    def fake_inference(news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                       user_category_mask, user_category_indices, news_graph_context):
        seen['inference'] = [tuple(t.shape) for t in (news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding,
                                                      user_graph, user_category_mask, user_category_indices, news_graph_context)]
        return news_graph_context, user_news_embedding[:, 0, :]

    def fake_forward(*a):
        seen['forward'] = [tuple(t.shape) for t in a]
        return a[0][:, 0, :], a[3][:, 0, :]
    model.graph_encoder.inference = fake_inference
    model.graph_encoder.forward = fake_forward
    Xh, Au = torch.randn(B, H, D), torch.zeros(B, n_u, n_u, dtype=torch.bool)
    Mc, ci = torch.ones(B, C1, dtype=torch.bool), torch.zeros(B, H, dtype=torch.int64)
    Xn, An, Mn = torch.randn(B, n_n, D), torch.zeros(B, n_n, n_n, dtype=torch.bool), torch.ones(B, n_n, dtype=torch.bool)
    c0 = torch.randn(B, D)
    out = model.inference(Xh, Au, Mc, ci, Xn, An, Mn, c0)                      # model.py:87-90 / util.py:68
    assert seen['inference'] == [(B, n_n, D), (B, n_n, n_n), (B, n_n), (B, H, D), (B, n_u, n_u), (B, C1), (B, H), (B, D)]
    assert torch.allclose(out, (Xh[:, 0, :] * c0).sum(1))
    # Model.forward: [bs, news_num, ...] candidates, user tensors expanded over news_num (model.py:54-77)
    bs, nn_ = 2, 3
    T = cfg.max_title_length
    logits = model(torch.zeros(bs, H, T, dtype=torch.long), torch.ones(bs, H, T), Au[:bs], Mc[:bs], ci[:bs],
                   torch.zeros(bs, nn_, n_n, T, dtype=torch.long), torch.ones(bs, nn_, n_n, T),
                   An[:bs].unsqueeze(1).expand(-1, nn_, -1, -1).contiguous(), Mn[:bs].unsqueeze(1).expand(-1, nn_, -1).contiguous())
    bn = bs * nn_
    assert seen['forward'] == [(bn, n_n, D), (bn, n_n, n_n), (bn, n_n), (bn, H, D), (bn, n_u, n_u), (bn, C1), (bn, H)]
    assert logits.shape == (bs, nn_)
