"""Generate tests/golden/*.pt by running the REAL reference modules (read-only tree at /root/reference) on CPU.

Run in the build container only:  python tests/golden/make_golden.py
The reference's own tests hold no numeric golden vectors for this path (SURVEY.md section 4), so these
fixtures are what pins the oracle (tests/test_oracle_vs_golden.py) and, on the GPU box where /root/reference
does not exist, the CUDA path (tests/test_gpu_*.py).  Inputs and weights are regenerated from seeds by
tests/helpers.py + audiocraft_b200/synth.py; only outputs are stored.
"""
import os
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import ref_import as R  # noqa: E402
from tests import helpers as H  # noqa: E402
from audiocraft_b200 import synth  # noqa: E402

warnings.filterwarnings('ignore')
torch.set_grad_enabled(False)


from oracle.ref_models import build_ref_encodec, build_ref_lm as _build_ref_lm  # noqa: E402


def build_ref_lm(cfg, sd, table):
    return _build_ref_lm(cfg, sd, table)


def golden_encodec(name, batch, length, wseed, xseed, full):
    cfg = synth.ENCODEC_CONFIGS[name]
    sd = synth.synth_encodec_state_dict(cfg, seed=wseed)
    m = build_ref_encodec(cfg, sd)
    x = H.audio_input(cfg, batch, length, xseed)
    codes, scale = m.encode(x)
    xin = m.preprocess(x)[0]
    latent = m.encoder(xin)
    wav = m.decode(codes, scale)
    qlat = m.decode_latent(codes)
    out = dict(name=name, batch=batch, length=length, wseed=wseed, xseed=xseed, codes=codes, scale=scale,
               x_head=x[..., :64].clone())
    if full:
        out.update(latent=latent, wav=wav, qlat=qlat)
    else:  # keep the fixture small: full codes, strided views of the float tensors
        out.update(latent=latent, wav_head=wav[..., :512].clone(), wav_stride=97,
                   wav_strided=wav[..., ::97].clone(), wav_len=wav.shape[-1])
    torch.save(out, os.path.join(H.GOLDEN_DIR, f'{name}.pt'))
    print(name, 'codes', tuple(codes.shape), 'wav', tuple(wav.shape))


def golden_lm(name, batch, t_text, T, wseed, cseed, steps_logits, topn=None):
    cfg = synth.lm_config(name)
    sd = synth.synth_lm_state_dict(cfg, seed=wseed)
    hid, mask, _ = H.lm_condition(cfg, sd, batch, t_text, cseed)
    table = {f'd{i}': (hid[i], mask[i]) for i in range(batch)}
    table['__null__'] = (torch.zeros(t_text, cfg['cond_dim']), torch.zeros(t_text, dtype=torch.long))
    m, CA = build_ref_lm(cfg, sd, table)
    conds = [CA(text={'description': f'd{i}'}) for i in range(batch)]
    out = dict(name=name, batch=batch, t_text=t_text, T=T, wseed=wseed, cseed=cseed)
    greedy = m.generate(None, conds, max_gen_len=T, use_sampling=False)
    out['greedy'] = greedy
    # teacher-forced logits along the greedy path: re-run with a hook on _sample_next_token's CFG-mixed logits
    logits = []
    orig = m._sample_next_token

    def spy(sequence, cfg_conditions, unconditional_state, use_sampling=False, temp=1.0, top_k=0, top_p=0.0,
            cfg_coef=None, cfg_coef_beta=None, two_step_cfg=None):
        B = sequence.shape[0]
        state = {k: v.clone() for k, v in m.get_streaming_state().items()}
        al = m(torch.cat([sequence, sequence], 0), conditions=[], condition_tensors=cfg_conditions)
        c, u = al.split(B, dim=0)
        coef = m.cfg_coef if cfg_coef is None else cfg_coef
        logits.append((u + (c - u) * coef)[:, :, -1, :].clone())
        m.set_streaming_state(state)
        return orig(sequence, cfg_conditions, unconditional_state, use_sampling, temp, top_k, top_p,
                    cfg_coef=cfg_coef, cfg_coef_beta=cfg_coef_beta, two_step_cfg=two_step_cfg)

    m._sample_next_token = spy
    greedy2 = m.generate(None, conds, max_gen_len=T, use_sampling=False)
    m._sample_next_token = orig
    assert (greedy2 == greedy).all()
    lg = torch.stack(logits[:steps_logits], 0)  # [steps,B,K,card]
    if topn is None:
        out['logits'] = lg
    else:
        tv, ti = lg.topk(topn, dim=-1)
        out['logits_top_v'], out['logits_top_i'] = tv, ti
    if topn is None:
        # sampled generations with torch's own generator (what the reference does, utils/utils.py:103)
        torch.manual_seed(11)
        out['sampled_topk'] = m.generate(None, conds, max_gen_len=T, use_sampling=True, top_k=10, temp=0.9)
        torch.manual_seed(12)
        out['sampled_topp'] = m.generate(None, conds, max_gen_len=T, use_sampling=True, top_k=0, top_p=0.8)
        torch.manual_seed(13)
        out['sampled_plain'] = m.generate(None, conds, max_gen_len=T, use_sampling=True, top_k=0, top_p=0.0, temp=1.3)
        out['continuation'] = m.generate(greedy[..., :5].clone(), conds, max_gen_len=T, use_sampling=False)
        # generate_unconditional: descriptions are None -> null condition rows, still doubled by CFG (genmodel.py:135-149)
        out['unconditional'] = m.generate(None, [CA(text={'description': None}) for _ in range(batch)],
                                          max_gen_len=T, use_sampling=False)
    torch.save(out, os.path.join(H.GOLDEN_DIR, f'{name}.pt'))
    print(name, 'greedy', tuple(greedy.shape))


def golden_patterns():
    pat = R.mod('modules.codebooks_patterns')
    out = {}
    for (K, T, delays) in [(4, 7, [0, 1, 2, 3]), (4, 1, [0, 1, 2, 3]), (8, 12, [0, 1, 2, 3, 4, 5, 6, 7]),
                           (3, 5, [0, 0, 2])]:
        p = pat.DelayedPatternProvider(K, delays=delays).get_pattern(T)
        g = torch.Generator()
        g.manual_seed(K * 100 + T)
        codes = torch.randint(0, 50, (2, K, T), generator=g)
        seq, idx, mask = p.build_pattern_sequence(codes, 99)
        back, idx2, mask2 = p.revert_pattern_sequence(seq, special_token=-1)
        out[(K, T, tuple(delays))] = dict(codes=codes, seq=seq, mask=mask, back=back, back_mask=mask2,
                                          first_step_T0=[p.get_first_step_with_timesteps(t) for t in range(T)])
    torch.save(out, os.path.join(H.GOLDEN_DIR, 'patterns.pt'))
    print('patterns', len(out))


def golden_sampling():
    utils = R.mod('utils.utils')
    g = torch.Generator()
    g.manual_seed(21)
    logits = torch.randn(6, 4, 2048, generator=g) * 2.0
    probs = torch.softmax(logits, -1)
    out = dict(seed=21)
    torch.manual_seed(31)
    out['top_k_250'] = utils.sample_top_k(probs.clone(), 250)
    torch.manual_seed(32)
    out['top_p_0.9'] = utils.sample_top_p(probs.clone(), 0.9)
    torch.manual_seed(33)
    out['plain'] = utils.multinomial(probs.clone(), 1)
    torch.save(out, os.path.join(H.GOLDEN_DIR, 'sampling.pt'))
    print('sampling ok')


def golden_stereo():
    """InterleaveStereoCompressionModel over the tiny mono codec (renormalize off), both interleavings."""
    enc = R.mod('models.encodec')
    cfg = dict(synth.ENCODEC_CONFIGS['encodec_tiny'])
    cfg['renormalize'] = False
    m = build_ref_encodec(cfg, synth.synth_encodec_state_dict(cfg, seed=1))
    cfg2 = dict(cfg)
    cfg2['channels'] = 2
    x = H.audio_input(cfg2, 2, 900, 9)
    out = dict(wseed=1, xseed=9, length=900, batch=2)
    for pt in (False, True):
        w = enc.InterleaveStereoCompressionModel(m, per_timestep=pt)
        codes, _ = w.encode(x)
        out[f'codes_pt{int(pt)}'] = codes
        out[f'wav_pt{int(pt)}'] = w.decode(codes, None)
        out[f'props_pt{int(pt)}'] = (w.num_codebooks, w.frame_rate, w.channels, w.cardinality, w.total_codebooks)
    torch.save(out, os.path.join(H.GOLDEN_DIR, 'encodec_tiny_stereo.pt'))


FULLSIZE_STEPS = [0, 1, 374, 749, 1124, 1499, 1502]   # teacher-forced steps kept (KV length = step + 1)


def golden_lm_fullsize(name, batch, t_text=16, T=1500, wseed=0, cseed=3, sseed=17, topn=32):
    """FULL-DEPTH released architectures at the benchmarked sequence length (VERDICT r1 item 1): one non-streaming causal
    forward of the reference LMModel (fp32, CPU) over a seeded delay-pattern sequence of T frames with the CFG rows
    [cond; null] = 2*batch, keeping the top-`topn` CFG-mixed logits at FULLSIZE_STEPS (LMModel.forward lm.py:221-268 +
    the mix of lm.py:393-399).  Weights / conditions / tokens are regenerated from seeds by the test."""
    import time
    t0 = time.time()
    cfg = synth.lm_config(name)
    sd = synth.synth_lm_state_dict(cfg, seed=wseed)
    _, _, cross = H.lm_condition(cfg, sd, batch, t_text, cseed)
    m, _ = build_ref_lm(cfg, sd, {'__null__': (torch.zeros(t_text, cfg['cond_dim']), torch.zeros(t_text, dtype=torch.long))})
    del sd
    seq = H.fullsize_sequence(cfg, batch, T, sseed)                     # [B, K, T + K] delay-pattern sequence
    S = seq.shape[-1]
    ct = {'description': (cross, torch.ones(cross.shape[:2], dtype=torch.long))}
    logits = m(torch.cat([seq, seq], 0)[..., :S - 1], conditions=[], condition_tensors=ct)   # [2B, K, S-1, card]
    c, u = logits.split(batch, dim=0)
    mixed = (u + (c - u) * cfg['cfg_coef'])[:, :, FULLSIZE_STEPS, :].permute(2, 0, 1, 3).contiguous()   # [n, B, K, card]
    tv, ti = mixed.topk(topn, dim=-1)
    out = dict(name=name, batch=batch, t_text=t_text, T=T, wseed=wseed, cseed=cseed, sseed=sseed, steps=FULLSIZE_STEPS,
               logits_top_v=tv, logits_top_i=ti.to(torch.int16), seq_head=seq[..., :16].clone(),
               cond_top_v=c[:, :, FULLSIZE_STEPS, :].permute(2, 0, 1, 3).gather(-1, ti), )
    torch.save(out, os.path.join(H.GOLDEN_DIR, f'{name}_full.pt'))
    print(name, 'fullsize logits', tuple(tv.shape), f'{time.time() - t0:.0f} s')


def golden_lm_fullsize_cuda(name, batch, items, t_text=16, T=1500, wseed=0, cseed=3, sseed=17, n_top=8, n_cols=56):
    """The reference's own CUDA path at the benchmarked shapes (needs a GPU): fp16 transformer under autocast, SDPA
    (audiocraft/models/loaders.py:115-118, genmodel.py:74-78), one causal forward over a seeded delay-pattern sequence of
    T frames with the CFG rows [cond; null] = 2*batch, weights generated on CUDA in fp16 exactly as the test regenerates
    them.  The full per-row logits ([7, 2*batch, K, card]) are too large to store, so the fixture keeps, for the batch
    items `items` (both CFG rows of each), the top-`n_top` logits of every row plus the logits at `n_cols` seeded columns,
    and for EVERY item the argmax and top-2 margin of the CFG-mixed logits.  The logits are fp16 values under autocast and
    are stored as such (lossless)."""
    import time
    t0 = time.time()
    dev = torch.device('cuda')
    cfg = synth.lm_config(name)
    sd = synth.synth_lm_state_dict(cfg, seed=wseed, device='cuda', dtype=torch.float16)
    w_head = sd['emb.0.weight'][:2, :16].cpu().clone()
    hid, mask = synth.synth_text_condition(cfg, batch, t_text, seed=cseed)
    from oracle import ref_models as RM
    ref, CA = RM.build_ref_lm(cfg, sd, RM.text_table(hid, mask, cfg['cond_dim']), device=dev, dtype=torch.float16)
    del sd
    seq = H.fullsize_sequence(cfg, batch, T, sseed).to(dev)
    S = seq.shape[-1]
    cc = RM.ref_cfg_conditions(ref, CA, batch)                           # {'description': ([2B,T,d] fp32, mask)}
    with torch.autocast('cuda', dtype=torch.float16):
        rl = ref(torch.cat([seq, seq], 0)[..., :S - 1], conditions=[], condition_tensors=cc)   # [2B,K,S-1,card]
    rl = rl[:, :, FULLSIZE_STEPS, :].float().permute(2, 0, 1, 3).contiguous().cpu()          # [n,2B,K,card]
    c, u = rl.split(batch, dim=1)
    rmix = u + (c - u) * cfg['cfg_coef']
    top2 = rmix.topk(2, dim=-1)
    rows = torch.tensor(list(items) + [batch + i for i in items])
    sub = rl[:, rows]
    tv, ti = sub.topk(n_top, dim=-1)
    g = torch.Generator()
    g.manual_seed(1000 + batch)
    cols = torch.randperm(cfg['card'], generator=g)[:n_cols].sort().values
    out = dict(name=name, batch=batch, t_text=t_text, T=T, wseed=wseed, cseed=cseed, sseed=sseed, steps=FULLSIZE_STEPS,
               w_head=w_head, cross_rowsum=cc['description'][0].float().sum(-1).cpu(), rows=rows,
               top_v=tv.half(), top_i=ti.to(torch.int16), cols=cols.to(torch.int16), cols_v=sub[..., cols].half(),
               mix_argmax=top2.indices[..., 0].to(torch.int16), mix_margin=top2.values[..., 0] - top2.values[..., 1])
    assert torch.equal(out['top_v'].float(), tv) and torch.equal(out['cols_v'].float(), sub[..., cols])
    torch.save(out, os.path.join(H.GOLDEN_DIR, f'{name}_cuda_autocast.pt'))
    print(name, 'reference CUDA autocast logits', tuple(rl.shape), 'kept rows', rows.tolist(), f'{time.time() - t0:.0f} s')


def golden_encodec_fullsize():
    """BASELINE config 1 at its real length (10 s = 240 000 samples at 24 kHz: codes [1, n_q, 750] for n_q = 8 and 32)
    and a [2, 1, 320000] slice of config 4 (32 kHz, 4 codebooks): codes from the reference (int16 to keep the fixture small)."""
    cfg = synth.ENCODEC_CONFIGS['encodec_24k']
    for n_q in (8, 32):
        c = dict(cfg)
        c['n_q'] = n_q
        sd = synth.synth_encodec_state_dict(c, seed=5)
        m = build_ref_encodec(c, sd)
        x = H.audio_input(c, 1, 240000, 6)
        codes, scale = m.encode(x)
        wav = m.decode(codes, scale)
        torch.save(dict(name='encodec_24k', n_q=n_q, batch=1, length=240000, wseed=5, xseed=6, codes=codes.to(torch.int16),
                        wav_stride=997, wav_strided=wav[..., ::997].clone(), wav_len=wav.shape[-1], x_head=x[..., :64].clone()),
                   os.path.join(H.GOLDEN_DIR, f'encodec_24k_10s_nq{n_q}.pt'))
        print('encodec_24k 10 s n_q', n_q, tuple(codes.shape))
    cfg = synth.ENCODEC_CONFIGS['encodec_32k']
    sd = synth.synth_encodec_state_dict(cfg, seed=7)
    m = build_ref_encodec(cfg, sd)
    x = H.audio_input(cfg, 2, 320000, 8)
    codes, scale = m.encode(x)
    wav = m.decode(codes, scale)
    torch.save(dict(name='encodec_32k', batch=2, length=320000, wseed=7, xseed=8, codes=codes.to(torch.int16),
                    wav_stride=997, wav_strided=wav[..., ::997].clone(), wav_len=wav.shape[-1], x_head=x[..., :64].clone()),
               os.path.join(H.GOLDEN_DIR, 'encodec_32k_10s.pt'))
    print('encodec_32k 2 x 10 s', tuple(codes.shape))


def golden_lm_rope():
    """Rotary positions (modules/rope.py:84-125, transformer.py:394-395, 632-637): lm_mini with positional_embedding
    'rope' and 'sin_rope' (positional_scale 0.75 so the scale blend is exercised).  Teacher-forced CFG-mixed logits from
    ONE non-streaming causal forward, and greedy generation in streaming mode with the reference's custom attention
    (memory_efficient=False) -- the mode tests/modules/test_rope.py:66-90 checks.  (With memory_efficient=True and the
    'torch' backend the reference's _apply_rope reads past_keys.shape[1], which is the HEAD count in the `b h t d` layout,
    transformer.py:304-305: streaming then rotates at the wrong offset; that quirk is not reproduced.)"""
    out = {}
    for pe in ('rope', 'sin_rope'):
        cfg = synth.lm_config('lm_mini')
        cfg['positional_embedding'], cfg['positional_scale'] = pe, 0.75
        sd = synth.synth_lm_state_dict(cfg, seed=3)
        B, t_text, T = 2, 5, 12
        hid, mask, cross = H.lm_condition(cfg, sd, B, t_text, 1)
        table = {f'd{i}': (hid[i], mask[i]) for i in range(B)}
        table['__null__'] = (torch.zeros(t_text, cfg['cond_dim']), torch.zeros(t_text, dtype=torch.long))
        m, CA = _build_ref_lm(cfg, sd, table, positional_embedding=pe, positional_scale=0.75, memory_efficient=False, custom=True)
        seq = H.fullsize_sequence(cfg, B, T, 5)
        ct = {'description': (cross, torch.ones(cross.shape[:2], dtype=torch.long))}
        lg = m(torch.cat([seq, seq], 0)[..., :-1], conditions=[], condition_tensors=ct)
        c, u = lg.split(B, dim=0)
        conds = [CA(text={'description': f'd{i}'}) for i in range(B)]
        out[pe] = dict(logits=(u + (c - u) * cfg['cfg_coef']).permute(2, 0, 1, 3).contiguous(),   # [S-1, B, K, card]
                       greedy=m.generate(None, conds, max_gen_len=T, use_sampling=False))
    out.update(batch=2, t_text=5, T=12, wseed=3, cseed=1, sseed=5, positional_scale=0.75)
    torch.save(out, os.path.join(H.GOLDEN_DIR, 'lm_mini_rope.pt'))
    print('lm_mini_rope ok')


def golden_two_step():
    """LMModel.generate(two_step_cfg=True) (lm.py:376-391, 497-503): two separate passes per step with their own streaming
    states, and the quirk that this branch mixes with self.cfg_coef, not the `cfg_coef` argument (lm.py:387)."""
    cfg = synth.lm_config('lm_mini')
    sd = synth.synth_lm_state_dict(cfg, seed=3)
    B, t_text, T = 2, 5, 12
    hid, mask, _ = H.lm_condition(cfg, sd, B, t_text, 1)
    table = {f'd{i}': (hid[i], mask[i]) for i in range(B)}
    table['__null__'] = (torch.zeros(t_text, cfg['cond_dim']), torch.zeros(t_text, dtype=torch.long))
    m, CA = _build_ref_lm(cfg, sd, table)
    conds = [CA(text={'description': f'd{i}'}) for i in range(B)]
    out = dict(batch=B, t_text=t_text, T=T, wseed=3, cseed=1,
               two_step=m.generate(None, conds, max_gen_len=T, use_sampling=False, two_step_cfg=True, cfg_coef=1.5),
               batched_coef_1p5=m.generate(None, conds, max_gen_len=T, use_sampling=False, two_step_cfg=False, cfg_coef=1.5),
               batched_default=m.generate(None, conds, max_gen_len=T, use_sampling=False))
    assert torch.equal(out['two_step'], out['batched_default'])   # the quirk: two-step ignores cfg_coef=1.5
    torch.save(out, os.path.join(H.GOLDEN_DIR, 'lm_mini_two_step.pt'))
    print('two_step ok; differs from coef 1.5:', not torch.equal(out['two_step'], out['batched_coef_1p5']))


if __name__ == '__main__':
    os.makedirs(H.GOLDEN_DIR, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] == 'two_step':
        golden_two_step()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'rope':
        golden_lm_rope()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'fullsize':
        golden_encodec_fullsize()
        golden_lm_fullsize('musicgen_medium', 8)
        golden_lm_fullsize('musicgen_large', 4)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'fullsize_cuda':   # on a CUDA device
        golden_lm_fullsize_cuda('musicgen_medium', 8, items=range(8))
        golden_lm_fullsize_cuda('musicgen_large', 32, items=[0, 5, 10, 15, 16, 21, 26, 31])
        sys.exit(0)
    golden_patterns()
    golden_sampling()
    golden_encodec('encodec_tiny', 2, 1234, 1, 2, full=True)
    golden_encodec('encodec_tiny_causal', 2, 777, 3, 4, full=True)
    golden_encodec('encodec_24k', 1, 24000, 5, 6, full=False)
    golden_encodec('encodec_32k', 1, 32000, 7, 8, full=False)
    golden_lm('lm_mini', 2, 5, 12, 3, 1, steps_logits=15)
    golden_lm('lm_tiny', 3, 4, 9, 4, 2, steps_logits=12)
    golden_lm('musicgen_small', 1, 6, 3, 9, 5, steps_logits=6, topn=32)
    golden_stereo()
    golden_lm_rope()
    golden_two_step()
