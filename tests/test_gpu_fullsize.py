"""Parity AT THE BENCHMARKED SIZES (VERDICT r1 item 1): full-depth MusicGen-medium / -large over a 1500-frame sequence
(KV length up to 1503), and EnCodec at 10 s, against

  (a) committed golden vectors the real reference produced on CPU in fp32 (tests/golden/make_golden.py fullsize), and
  (b) committed golden vectors of the reference's OWN CUDA path on a B200 -- fp16 transformer under autocast, SDPA
      (audiocraft/models/loaders.py:115-118, genmodel.py:74-78) -- i.e. the arithmetic the reference really runs for
      configs 2/3/5, not an emulation of it (tests/golden/make_golden.py fullsize_cuda).

Tolerances (fp16 weights and fp16 GEMM outputs on |logits| ~ 20, where fp16 spacing alone is 1.6e-2):
  per-row logits vs the reference CUDA path: atol 5e-2;  CFG-mixed logits (u + 3 (c - u) amplifies both branches'
  error ~5x) vs fp32 CPU golden: atol 1.2e-1 and the top-1 token must agree wherever the reference's own top-2 margin
  exceeds that.  EnCodec codes: exact, except where the reference's own best/second-best distance gap is below fp32
  summation noise (reported)."""
import os

import pytest
import torch

from tests import helpers as H
from audiocraft_b200 import synth

pytestmark = pytest.mark.gpu


def _golden(name):
    p = os.path.join(H.GOLDEN_DIR, name)
    if not os.path.exists(p):
        pytest.skip(f'{name} not generated')
    return torch.load(p, weights_only=False)


def _lm(name, sd):
    from audiocraft_b200.lm import LMModel
    return LMModel(sd, synth.lm_config(name), None, None, 'cuda')


@pytest.mark.parametrize('name', ['musicgen_medium', 'musicgen_large'])
def test_fulldepth_logits_match_reference_cpu_golden(name):
    g = _golden(f'{name}_full.pt')
    cfg = synth.lm_config(name)
    sd = synth.synth_lm_state_dict(cfg, seed=g['wseed'])                # CPU generator: the weights the golden was made with
    _, _, cross = H.lm_condition(cfg, sd, g['batch'], g['t_text'], g['cseed'])
    seq = H.fullsize_sequence(cfg, g['batch'], g['T'], g['sseed'])
    assert torch.equal(seq[..., :16], g['seq_head'])
    m = _lm(name, sd)
    del sd
    S = seq.shape[-1]
    lg = m.teacher_forced_logits(seq, cross, cfg['cfg_coef'], n_steps=S - 1, keep=g['steps']).cpu()   # [n,B,K,card]
    ti = g['logits_top_i'].long()
    got = lg.gather(-1, ti)
    err = (got - g['logits_top_v']).abs()
    print(f'{name}: full depth, KV up to {S - 1}: max |CFG-mixed logit diff| vs fp32 reference per kept step:',
          [round(float(e), 4) for e in err.amax(dim=(1, 2, 3))])
    assert float(err.max()) < 1.2e-1
    margin = g['logits_top_v'][..., 0] - g['logits_top_v'][..., 1]
    agree = lg.argmax(-1) == ti[..., 0]
    assert bool(agree[margin > 1.2e-1].all()), 'top-1 token differs from the reference outside a near-tie'
    print(f'   top-1 agreement {agree.float().mean():.4f} ({int((margin <= 1.2e-1).sum())} near-ties of {margin.numel()})')


@pytest.mark.parametrize('name,batch', [('musicgen_medium', 8), ('musicgen_large', 32)])
def test_fulldepth_logits_match_reference_cuda_autocast(name, batch):
    """BENCH shapes exactly: medium rows 16 (config 3), large rows 64 (config 5), S = 1504, against the reference's own
    CUDA path (fp16 autocast, SDPA) stored by tests/golden/make_golden.py fullsize_cuda: per-row logits of the stored rows
    at their top entries and at seeded columns, and the CFG-mixed argmax of every item."""
    g = _golden(f'{name}_cuda_autocast.pt')
    assert g['batch'] == batch
    cfg = synth.lm_config(name)
    sd = synth.synth_lm_state_dict(cfg, seed=g['wseed'], device='cuda', dtype=torch.float16)
    assert torch.equal(sd['emb.0.weight'][:2, :16].cpu(), g['w_head']), 'seeded CUDA weights are not the ones the golden was made with'
    _, _, cross = H.lm_condition(cfg, sd, batch, g['t_text'], g['cseed'])  # [cond; null] rows, as the reference's condition provider
    torch.testing.assert_close(cross.sum(-1), g['cross_rowsum'], rtol=0, atol=1e-3)
    seq = H.fullsize_sequence(cfg, batch, g['T'], g['sseed']).cuda()
    S = seq.shape[-1]
    m = _lm(name, sd)
    del sd
    mixed, raw = m.teacher_forced_logits(seq, cross, cfg['cfg_coef'], n_steps=S - 1, keep=g['steps'], raw=True)
    raw = raw.cpu()[:, g['rows']]                                          # [n, stored rows, K, card]
    err_top = (raw.gather(-1, g['top_i'].long()) - g['top_v'].float()).abs()
    err_cols = (raw[..., g['cols'].long()] - g['cols_v'].float()).abs()
    err = torch.maximum(err_top.amax(-1), err_cols.amax(-1))
    print(f'{name} rows={2 * batch}: max |per-row logit diff| vs the reference CUDA autocast path per kept step:',
          [round(float(e), 4) for e in err.amax(dim=(1, 2))], ' mean', round(float(err_cols.mean()), 5))
    assert float(err.max()) < 5e-2
    margin = g['mix_margin']
    agree = mixed.argmax(-1).cpu() == g['mix_argmax'].long()
    print(f'   greedy token agreement with the reference: {agree.float().mean():.4f}; outside near-ties (margin > 0.15): '
          f'{agree[margin > 0.15].float().mean():.4f}')
    assert bool(agree[margin > 0.15].all())


@pytest.mark.parametrize('fixture', ['encodec_24k_10s_nq8.pt', 'encodec_24k_10s_nq32.pt', 'encodec_32k_10s.pt'])
def test_encodec_10s_codes_match_reference_golden(fixture):
    from audiocraft_b200.encodec import EncodecModel
    g = _golden(fixture)
    cfg = dict(synth.ENCODEC_CONFIGS[g['name']])
    if 'n_q' in g:
        cfg['n_q'] = g['n_q']
    sd = synth.synth_encodec_state_dict(cfg, seed=g['wseed'])
    x = H.audio_input(cfg, g['batch'], g['length'], g['xseed'])
    assert torch.equal(x[..., :64], g['x_head'])
    m = EncodecModel(sd, cfg, 'cuda')
    codes, scale = m.encode(x.cuda())
    want = g['codes'].long()
    assert codes.shape == want.shape
    same = (codes.cpu() == want)
    frames_ok = same.all(dim=1).float().mean().item()
    print(f'{fixture}: codes {tuple(codes.shape)} exact for {same.float().mean():.6f} of indices, {frames_ok:.6f} of frames')
    if not bool(same.all()):   # only the FIRST differing codebook of a frame is judged (later ones follow from it)
        from oracle import encodec_oracle as EO
        o = EO.EncodecOracle(sd, cfg)
        lat = o.encode_latent(o.preprocess(x)[0])
        ocodes, margins = EO.rvq_encode(lat, EO.codebooks_of(sd, cfg['n_q']), return_margin=True)
        assert torch.equal(ocodes, want), 'oracle and reference golden disagree'
        neq = ~same
        first = neq.int().cumsum(1).eq(1) & neq
        gaps = margins[first]
        print(f'   {int(first.sum())} near-tie code flips, reference margins {gaps.tolist()[:8]}')
        assert (gaps.abs() < 1e-4).all(), 'RVQ index mismatch with a clear margin'
    wav = m.decode(want.cuda(), None).cpu()
    assert wav.shape[-1] == g['wav_len']
    torch.testing.assert_close(wav[..., ::g['wav_stride']], g['wav_strided'], rtol=0, atol=1e-4)
