"""Operands loaded before griddepcontrol.wait in the decode step: the cross-attention text K / V, the self-attention ring stages
of cache positions < pos, and the GEMM activation block staged in shared memory right after the wait.  None of it changes an
operation or a summation order, so every comparison here is bit for bit.  Default vs ACB_LM_FT32=0 tiles at MusicGen-medium
widths, rows 16, is test_gpu_lm.py::test_ft32_tiles_equal_16_feature_tiles."""
import pytest
import torch

from tests import helpers as H
from audiocraft_b200 import synth

pytestmark = pytest.mark.gpu


def _model(name, wseed):
    from audiocraft_b200.lm import LMModel
    cfg = synth.lm_config(name)
    sd = synth.synth_lm_state_dict(cfg, seed=wseed)
    return cfg, sd, LMModel(sd, cfg, None, None)


def test_prewait_ring_equals_register_attention_across_stage_boundary(monkeypatch):
    """lm_attn2_kernel fills its first 7 ring stages (7 x 32 positions) before the wait and loads position pos after it;
    ACB_LM_ATTN=v1 loads everything after the wait.  KV lengths straddle 224 and reach 1500 at medium widths, rows 16."""
    cfg, sd, m = _model('lm_medium_2l', 5)
    B, T = 8, 1500
    _, _, cross = H.lm_condition(cfg, sd, B, 6, 1)
    seq = torch.randint(0, cfg['card'], (B, 4, T + 4), generator=torch.Generator().manual_seed(2))
    keep = [0, 1, 222, 223, 224, T - 1]      # KV lengths 1, 2, 223, 224, 225, 1500
    a = m.teacher_forced_logits(seq, cross, 3.0, n_steps=T, keep=keep).cpu()
    monkeypatch.setenv('ACB_LM_ATTN', 'v1')
    b = m.teacher_forced_logits(seq, cross, 3.0, n_steps=T, keep=keep).cpu()
    assert torch.isfinite(a).all()
    assert torch.equal(a, b), f'max diff {(a - b).abs().max():.3e}'


def test_direct_steps_equal_graph_steps():
    """The same step sequence through directly enqueued steps (first kernel launched without PDL) and through the
    captured graph gives identical raw logits."""
    cfg, sd, m = _model('lm_medium_2l', 7)
    B, T = 8, 12
    _, _, cross = H.lm_condition(cfg, sd, B, 6, 3)
    rows = 2 * B
    graph = []
    m.generate(None, [], num_samples=B, max_gen_len=T, use_sampling=False, cross_attention_src=cross,
               callback=lambda *_: graph.append(m._bufs['logits'][:rows].clone()))
    graph = torch.stack(graph).cpu()
    _, direct = m.teacher_forced_logits(m.last_sequence, cross, cfg['cfg_coef'], raw=True)
    direct = direct.cpu().reshape(direct.shape[0], rows, -1)
    assert graph.shape[0] == direct.shape[0]
    assert torch.equal(graph.reshape(direct.shape), direct)


@pytest.mark.parametrize('streaming', [False, True])
def test_second_condition_equals_fresh_model(streaming):
    """Two generations on one model with different text conditions (different lengths, one above 32 positions): each
    equals a fresh model's run, so no pre-wait read of the cross K / V sees the previous condition."""
    cfg, sd, m = _model('lm_medium_2l', 9)
    B, T = 8, 10
    conds = [H.lm_condition(cfg, sd, B, 6, 4)[2], H.lm_condition(cfg, sd, B, 37, 5)[2]]
    seq = torch.randint(0, cfg['card'], (B, 4, T), generator=torch.Generator().manual_seed(4))

    def run(model, cross):
        if streaming:
            model.streaming_begin(B, cross, max_len=T)
            return torch.stack([model.streaming_step(seq[..., i]).clone() for i in range(T)]).cpu()
        return model.generate(None, [], num_samples=B, max_gen_len=T, use_sampling=False, cross_attention_src=cross).cpu()

    got = [run(m, c) for c in conds]
    for c, g in zip(conds, got):
        want = run(_model('lm_medium_2l', 9)[2], c)
        assert torch.equal(g, want)
    assert not torch.equal(got[0], got[1])
