"""CPU tests: the C-ABI library loads and exports every symbol the header declares, the host logic (padding geometry,
delay pattern, conditioning plumbing, loaders) matches the oracle / reference golden vectors, and the product path
fails loudly without a GPU (no CPU fallback)."""
import os
import re

import pytest
import torch

from tests import helpers as H
from audiocraft_b200 import synth
from oracle import encodec_oracle as EO, lm_oracle as LO


def test_library_exports_every_declared_symbol():
    from audiocraft_b200 import _lib, build
    build.build()
    L = _lib.lib()
    header = open(os.path.join(H.ROOT, 'include', 'audiocraft_b200.h')).read()
    declared = set(re.findall(r'\b(acb_[a-z0-9_]+)\s*\(', header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(L, name), name
    assert L.acb_version() >= 100
    assert L.acb_lm_rows_pad(1) == 16 and L.acb_lm_rows_pad(16) == 16 and L.acb_lm_rows_pad(17) == 32 and L.acb_lm_rows_pad(64) == 64
    assert L.acb_lstm_state_bytes(2, 8) == (2 * 32 * 8 + 64) * 4      # h double buffer for max(batch, 32) item slots + barrier counters
    assert L.acb_lstm_state_bytes(40, 8) == (2 * 40 * 8 + 64) * 4


def test_fused_residual_block_routing():
    """Which SEANet residual blocks go to acb_resblock (host rule in EncodecModel._fused_block, no GPU needed): the 32 kHz model's
    identity-skip blocks at 64 / 128 / 256 channels yes; 32 / 512 channels, conv-shortcut blocks and the all-FMA precision no."""
    from types import SimpleNamespace
    from audiocraft_b200 import _lib
    from audiocraft_b200.encodec import EncodecModel, encodec_layers
    L = _lib.lib()
    assert [L.acb_resblock_supported(c, 3, 1) for c in (32, 64, 128, 256, 512)] == [0, 1, 1, 1, 0]
    assert L.acb_resblock_supported(64, 3, 4) == 1 and L.acb_resblock_supported(64, 3, 5) == 0 and L.acb_resblock_supported(64, 5, 1) == 0
    stub = SimpleNamespace(_fuse_blocks=True, _lib=L)

    def fused(cfg_name, prec):
        plan = encodec_layers(synth.ENCODEC_CONFIGS[cfg_name])
        out = []
        for part in ('encoder', 'decoder'):
            layers, have_shortcut = plan[part], False
            for i, lay in enumerate(layers):
                if lay['kind'] == 'conv' and lay['res'] == 'shortcut':
                    have_shortcut = True
                if not have_shortcut and EncodecModel._fused_block(stub, layers, i, prec, 4000):
                    out.append(layers[i + 1]['cout'])
                if lay['kind'] == 'conv' and lay['res'] == 'out':
                    have_shortcut = False
        return out

    assert fused('encodec_32k', _lib.CONV_T6_AUTO) == [64, 128, 256, 256, 128, 64]      # encoder then decoder; the 512-channel blocks stay two kernels
    assert fused('encodec_32k', _lib.CONV_TF32X3) == [64, 128, 256, 256, 128, 64]
    assert fused('encodec_32k', _lib.CONV_FP32) == []                                     # 'fp32' = every convolution on FMA
    assert fused('encodec_24k', _lib.CONV_T6_AUTO) == [64, 128, 256, 256, 128, 64]       # 32 -> 512 channels: the 32- and 512-channel blocks stay two kernels
    plan = encodec_layers(dict(synth.ENCODEC_CONFIGS['encodec_32k'], true_skip=False))      # conv shortcut (the HF EnCodec layout): never fused
    assert any(lay.get('res') == 'shortcut' for lay in plan['encoder'])
    stub._fuse_blocks = False
    assert fused('encodec_32k', _lib.CONV_T6_AUTO) == []


def test_sass_is_sm100a():
    import subprocess
    from audiocraft_b200 import _lib, build
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), 'cuobjdump')   # the toolkit that built the library, on PATH or not
    out = subprocess.run([cuobjdump, '-lelf', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert 'sm_100a' in out, out


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from audiocraft_b200.encodec import EncodecModel
    from audiocraft_b200.lm import LMModel
    cfg = synth.ENCODEC_CONFIGS['encodec_tiny']
    with pytest.raises(RuntimeError, match='no CPU'):
        EncodecModel(synth.synth_encodec_state_dict(cfg, 0), cfg)
    lcfg = synth.lm_config('lm_tiny')
    with pytest.raises(RuntimeError, match='no CPU'):
        LMModel(synth.synth_lm_state_dict(lcfg, 0), lcfg)


def test_conv_geometry_matches_oracle():
    from audiocraft_b200.encodec import conv_geometry, convtr_geometry
    for (k, s, d) in [(7, 1, 1), (3, 1, 1), (3, 1, 2), (3, 1, 4), (8, 4, 1), (10, 5, 1), (16, 8, 1), (4, 2, 1), (1, 1, 1)]:
        for causal in (False, True):
            for L in (1, 2, 3, 5, 8, 49, 50, 640, 641, 32000):
                left, right = EO.conv_paddings(L, k, s, d, causal)
                x = torch.arange(L, dtype=torch.float32).view(1, 1, L)
                padded = EO.pad1d(x, left, right, 'reflect')
                gl, tv, tout = conv_geometry(L, k, s, d, causal, True)
                assert gl == left
                assert tout == (padded.shape[-1] - ((k - 1) * d + 1)) // s + 1
                # the kernel's index rule reproduces pad1d exactly
                idx = torch.arange(padded.shape[-1]) - left
                idx = torch.where(idx < 0, -idx, idx)
                idx = torch.where(idx >= tv, 2 * (tv - 1) - idx, idx)
                val = torch.where((idx >= 0) & (idx < L), x[0, 0][idx.clamp(0, L - 1)], torch.zeros(()))
                assert torch.equal(val, padded[0, 0]), (k, s, d, causal, L)
    for (k, s) in [(4, 2), (6, 3), (8, 4), (10, 5), (16, 8)]:
        for causal, ratio in [(False, 1.0), (True, 1.0), (True, 0.5), (True, 0.0)]:
            tl, tout = convtr_geometry(13, k, s, causal, ratio)
            y = EO.sconvtr1d(torch.randn(1, 1, 13), torch.randn(1, 1, k), torch.zeros(1), s, causal, ratio)
            assert tout == y.shape[-1] == 13 * s


def test_layer_plan_covers_reference_keys():
    """The layer plan enumerates exactly the reference's state_dict keys (checked against golden-tested synth dicts)."""
    for name, cfg in synth.ENCODEC_CONFIGS.items():
        sd = synth.synth_encodec_state_dict(cfg, 0)
        plan = synth.encodec_layers(cfg)
        prefixes = [l['prefix'] for l in plan['encoder'] + plan['decoder']]
        for k in sd:
            assert k.startswith('quantizer.') or any(k.startswith(p) for p in prefixes), k
    enc = synth.encodec_layers(synth.ENCODEC_CONFIGS['encodec_32k'])['encoder']
    idx = sorted({int(l['prefix'].split('.')[2]) for l in enc})
    assert idx == [0, 1, 3, 4, 6, 7, 9, 10, 12, 13, 15]   # SURVEY.md section 8b


def test_patterns_match_reference_golden():
    from audiocraft_b200.patterns import DelayedPatternProvider
    g = torch.load(os.path.join(H.GOLDEN_DIR, 'patterns.pt'), weights_only=False)
    for (K, T, delays), ref in g.items():
        p = DelayedPatternProvider(K, delays=list(delays)).get_pattern(T)
        seq, _, mask = p.build_pattern_sequence(ref['codes'], 99)
        assert torch.equal(seq, ref['seq']) and torch.equal(mask, ref['mask'])
        back, _, bmask = p.revert_pattern_sequence(seq, special_token=-1)
        assert torch.equal(back, ref['back']) and torch.equal(bmask, ref['back_mask'])
        assert [p.get_first_step_with_timesteps(t) for t in range(T)] == ref['first_step_T0']
        # partially filled codes (generation in progress)
        part = ref['codes'].clone()
        part[..., T // 2:] = -1
        s2, m2 = LO.build_delay_sequence(part, list(delays), 99)
        s3, _, m3 = p.build_pattern_sequence(part, 99)
        assert torch.equal(s2, s3) and torch.equal(m2, m3)


def test_conditioning_plumbing():
    from audiocraft_b200.conditioners import (ConditionFuser, ConditioningAttributes, ConditioningProvider,
                                              PrecomputedTextConditioner, nullify_all)
    from audiocraft_b200.loaders import synthetic_text_encoder
    cfg = synth.lm_config('lm_mini')
    enc = synthetic_text_encoder(cfg, t_text=6)
    prov = ConditioningProvider({'description': PrecomputedTextConditioner(cfg['cond_dim'], cfg['dim'], enc)})
    conds = [ConditioningAttributes(text={'description': 'a b c'}), ConditioningAttributes(text={'description': None})]
    allc = conds + nullify_all(conds)
    assert conds[0].text['description'] == 'a b c'  # nullify works on a copy
    tens = prov(prov.tokenize(allc))
    emb, mask = tens['description']
    assert emb.shape == (4, 6, cfg['dim']) and mask.shape == (4, 6)
    assert mask[0].sum() == 4 and mask[1:].sum() == 0
    assert emb[1:].abs().max() == 0 and emb[0, :4].abs().sum() > 0 and emb[0, 4:].abs().max() == 0
    cross = ConditionFuser({'cross': ['description']}).cross_source(tens)
    assert cross is emb
    with pytest.raises(NotImplementedError):
        ConditionFuser({'prepend': ['description']})
    with pytest.raises(AssertionError):
        prov.tokenize(['not attributes'])


def test_loaders_fail_loudly():
    from audiocraft_b200 import loaders
    with pytest.raises(FileNotFoundError):
        loaders.load_compression_model('facebook/encodec_32khz')
    with pytest.raises(FileNotFoundError):
        loaders.load_musicgen('facebook/musicgen-medium')


def test_shard_bounds():
    from audiocraft_b200.dist import shard_bounds
    for n in (1, 7, 8, 9, 256):
        for world in (1, 2, 3, 8):
            spans = [shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
