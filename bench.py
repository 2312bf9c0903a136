"""bench.py -- MusicGen-medium text-conditioned 30 s generation, batch 8 per GPU (BASELINE.json configs[2]), the
configuration the headline metric `audio-sec/sec` is quoted on; it fits one B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--duration 30] [--batch 8]
                  [--scaling weak|strong] [--scale small|medium|large] [--workload musicgen|encodec] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...

Defaults = BASELINE configs[2] with `--batch` items PER GPU (`scaling: weak`, as the contract prescribes for a path that shards
by independent items).  `--scaling strong` splits `--batch` items over the ranks instead (configs[2] read literally: batch 8 over
1-8 GPUs = 8/4/2/1 items per GPU) and gathers the waveforms with NCCL inside the timed region.  `--scale large --batch 32
--scaling strong` is configs[4]; `--workload encodec --batch 256 --scaling strong` is configs[3] (EnCodec 32 kHz encode+decode
throughput, its own metric / roofline / CPU baseline).

One "step" = one full pass of the hot path over one batch: LMModel.generate (T+3 decode steps, CFG rows = 2B) followed
by EnCodec decode of the tokens to audio.  `value` = audio seconds produced by all ranks / max-over-ranks device time,
inputs (condition tensors) resident in HBM.  `e2e` = the same through the public MusicGen.generate(descriptions) call
with host inputs (text-encoder states pinned on the host, copied inside the timed region) and the waveform read back.
Weights are seeded random (no checkpoints offline), inputs synthetic.

`--dump-outputs DIR` writes what the last timed step returned on rank 0 as DIR/<name>.npy (float32): `tokens` [B, K, T] and
`wav` [B, 1, samples] for MusicGen, `codes` and `wav` for EnCodec (see dump_outputs for outputs over 64 MB).  Inputs, weights
and sampling seeds are fixed, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the reference's OWN code on the box's host cores: the unmodified package installed under
baseline/_ref (baseline/install_ref.sh; it ships with the snapshot), driven through oracle/ref_import.py's third-party
stubs by baseline/reference_arm.py.  One "step" of that arm is one bounded sample of the same workload (a few decode
steps of LMModel.generate's loop at KV length 1 and at the final KV length + the EnCodec decode of 1 s of tokens),
integrated to the full pass; `ms_per_step` is the sample's wall time.  The b200 line carries the same measurement as
`cpu_baseline` and, as `reference_gpu`, the reference's CUDA path (fp16 autocast, SDPA, eager) timed over full passes on
the same GPU -- the competitor north_star names.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MusicGen-medium audio-sec/sec @30s gen"
UNIT = "audio-s/s"


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j['hbm_gbs'], source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (recipe in B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '200',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons),
                    samples=len(sm))


def dist_setup(n):
    if n <= 1:
        return 0, 1
    import torch.distributed as dist
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    local = int(os.environ.get('LOCAL_RANK', rank))
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
    if torch.cuda.is_available():
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    else:
        dist.init_process_group('gloo')
    return rank, world


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict):
    """Write each tensor of `arrays` as `path`/<name>.npy in float32.  When together they exceed DUMP_LIMIT_BYTES, every
    array is flattened and keeps the same fraction of its elements, at sorted positions drawn from a fixed seed: the sample
    is the same in every run, so two dumps still compare element for element."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().to('cpu', torch.float32) for k, v in arrays.items()}
    total = sum(v.numel() for v in arrays.values())
    budget = (DUMP_LIMIT_BYTES - 1024 * len(arrays)) // 4       # float32 elements; 1 KB per file for the .npy header
    for name, v in arrays.items():
        if total > budget:
            n = v.numel() * budget // total
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
            v = v.reshape(-1)[idx]
        np.save(os.path.join(path, f'{name}.npy'), v.numpy())


def encodec_roofline(samples: int, ms: float):
    """SURVEY.md section 8d for EnCodec-32k encode+decode: 4 822 B/sample when every layer reads its input and writes its
    output once (fp32, ELU / residual / padding fused) and 486 kFLOP/sample.  With tensor-core convolutions the per-layer design
    is HBM-bound (101 FLOP/B < the ridge), so the HBM figure is the binding one; the tensor figure is reported beside it."""
    pj = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))) if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else {}
    hbm = pj.get('hbm_gbs', 6650.0)
    tf = pj.get('bf16_tflops_sustained', 1400.0)
    gbs = samples * 4822 / (ms / 1e3) / 1e9
    tfl = samples * 486e3 / (ms / 1e3) / 1e12
    return dict(bound='hbm', achieved=round(gbs, 1), peak=hbm, unit='GB/s', frac=round(gbs / hbm, 4), traffic=None,
                algorithmic_bytes_per_sample=4822, peak_source='measured (MEASURED_PEAKS.json)' if pj else 'fallback (B200_PROFILING.md)',
                tensor=dict(achieved=round(tfl, 2), peak=tf, unit='TFLOP/s (fp32-equivalent work vs the measured dense bf16 peak)',
                            frac=round(tfl / tf, 4), flop_per_sample=486000))


def run_encodec(args):
    """BASELINE configs[3]: EnCodec 32 kHz, 4 codebooks, `--batch` x 10 s encode + decode, items split over the ranks
    (`--scaling strong`, 256 items -> 32 per GPU on 8) or `--batch` items per rank (weak)."""
    rank, world = dist_setup(args.gpus)
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a CUDA device; there is no CPU fallback"
    dev = torch.device('cuda', torch.cuda.current_device())
    from audiocraft_b200.loaders import load_compression_model
    from audiocraft_b200.dist import shard_bounds
    strong = args.scaling == 'strong'
    if strong:
        a_, b_ = shard_bounds(args.batch, rank, world)
        B = b_ - a_
    else:
        B = args.batch
    total_items = args.batch if strong else args.batch * world
    n_samp = int(10.0 * 32000)
    cm = load_compression_model('synthetic/encodec_32k', dev, seed=1)
    g = torch.Generator().manual_seed(7 + rank)
    x_host = (torch.randn(B, 1, n_samp, generator=g) * 0.1).pin_memory()
    x_dev = x_host.to(dev)
    CH = 32                                           # items per launch chain: bounds the activation memory ([32, 64, 320000] fp32 = 2.6 GB per layer)

    def step_device():
        outs = []
        for i in range(0, B, CH):
            codes, scale = cm.encode(x_dev[i:i + CH])
            outs.append((codes, cm.decode(codes, scale)))
        return outs

    def step_e2e():
        y = torch.empty((B, 1, n_samp), dtype=torch.float32, pin_memory=True)
        for i in range(0, B, CH):
            xb = x_host[i:i + CH].to(dev, non_blocking=True)
            codes, scale = cm.encode(xb)
            w = cm.decode(codes, scale)
            y[i:i + CH].copy_(w[..., :n_samp], non_blocking=True)
        return y

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()

    def timed(fn, n):
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms, out

    for _ in range(args.warmup):
        step_device()
    l0 = cm.launches
    with ClockSampler(torch.cuda.current_device()) as clk:
        ms, outs = timed(step_device, args.steps)
    clocks = clk.summary()
    launches = (cm.launches - l0) // args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(codes=torch.cat([c.cpu() for c, _ in outs]),
                                             wav=torch.cat([w.cpu() for _, w in outs])))
    del outs
    ms_e2e, _ = timed(step_e2e, max(1, min(args.steps, 3)))
    n_e2e = max(1, min(args.steps, 3))
    samples_step = total_items * n_samp
    value = samples_step * args.steps / (ms / 1e3) / 1e6
    cpu_baseline = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu:
        from baseline import reference_arm as RA
        if RA.available():
            cpu_baseline = RA.cpu_encodec_baseline(1, 10.0)
    if rank == 0:
        emit(dict(metric='EnCodec 32kHz encode+decode MSamples/sec', value=round(value, 2), unit='MSamples/s', n_gpus=world,
                  steps=args.steps, warmup=args.warmup, ms_per_step=round(ms / args.steps, 2), higher_is_better=True,
                  scaling=args.scaling, vs_baseline=None, dtype='f32', data='synthetic',
                  config=dict(workload=f'EnCodec 32 kHz, 4 codebooks: encode + decode of {total_items} x 10 s mono, {B} items on this rank '
                                       f'(launch chains of {CH} items); encoder fp32-accurate (index-exact), decoder 3xTF32 on tcgen05',
                              global_batch=total_items, seq_len=n_samp, parallelism=f'dp{world} (items split, no collective)',
                              l2=f'inputs larger than L2: every layer of a {CH}-item chain reads / writes 0.3-2.6 GB'),
                  clocks=clocks,
                  e2e=dict(value=round(samples_step * n_e2e / (ms_e2e / 1e3) / 1e6, 2), unit='MSamples/s',
                           h2d_bytes_per_step=B * n_samp * 4, d2h_bytes_per_step=B * n_samp * 4),
                  gpu_launches=launches * args.steps,
                  roofline=encodec_roofline(B * n_samp, ms / args.steps), cpu_baseline=cpu_baseline))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def algorithmic_bytes(lm, rows, S):
    """SURVEY.md section 8d: per decode step W_step + rows*t*kv_tok (read) + rows*kv_tok (write), fp16."""
    kv_tok = 2 * lm.dim * 2 * lm.num_layers
    w = lm.weight_bytes_per_step
    total = 0
    for t in range(1, S):  # step at position t-1 attends t keys
        total += w + rows * t * kv_tok + rows * kv_tok
    return w, kv_tok, total


def run_b200(args):
    rank, world = dist_setup(args.gpus)
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a CUDA device; there is no CPU fallback"
    dev = torch.device('cuda', torch.cuda.current_device())
    from audiocraft_b200 import _lib
    from audiocraft_b200.loaders import load_musicgen
    import ctypes as C
    torch.manual_seed(1234 + rank)
    strong = args.scaling == 'strong'
    if strong:
        from audiocraft_b200.dist import shard_bounds
        lo_, hi_ = shard_bounds(args.batch, rank, world)
        B = hi_ - lo_
        assert B >= 1, f'--scaling strong: batch {args.batch} < {world} ranks'
    else:
        B = args.batch
    dur = args.duration
    total_items = args.batch if strong else args.batch * world
    mg = load_musicgen(f'synthetic/{args.scale}', device=dev, seed=0)
    mg.set_generation_params(duration=dur, use_sampling=True, top_k=250, temperature=1.0, cfg_coef=3.0)
    lm, cm = mg.lm, mg.compression_model
    T = int(dur * mg.frame_rate)
    S = T + 3 + 1
    descriptions = [f"synthetic prompt number {i} for rank {rank} with a few more words" for i in range(B)]
    # device-resident inputs for `value`: the fused condition tensor [2B, T_text, d]
    from audiocraft_b200.conditioners import ConditioningAttributes
    attrs = [ConditioningAttributes(text={'description': d}) for d in descriptions]
    cross = lm._prepare_conditions(attrs, False, None).contiguous()
    # host inputs for `e2e`: the text-encoder hidden states live in PINNED host memory and are handed to the public call
    # MusicGen.generate(descriptions) by the conditioner's encoder hook (the frozen T5 is outside the hot path): the H2D copy
    # happens inside generate(), in the timed region, and the waveform is read back to the host.
    cond_mod = lm.condition_provider.conditioners['description']
    synth_enc = cond_mod.encoder
    table = {}
    for dsc in descriptions + [""]:
        h_, m_ = synth_enc([dsc])
        table[dsc] = (h_[0].pin_memory(), m_[0].pin_memory())

    def pinned_encoder(entries):
        return torch.stack([table[e][0] for e in entries]).pin_memory(), torch.stack([table[e][1] for e in entries]).pin_memory()

    hid, msk = pinned_encoder(descriptions + [""] * B)
    h2d_bytes = hid.numel() * 4 + msk.numel() * 8

    def step_device():
        tokens = lm.generate(None, [], num_samples=B, max_gen_len=T, cross_attention_src=cross, **mg.generation_params)
        wav = mg.generate_audio(tokens)
        if strong and world > 1:   # configs[2] read literally: one batch over the ranks, the audio gathered on every rank
            from audiocraft_b200.dist import gather_batch
            wav = gather_batch(wav, args.batch)
        return tokens, wav

    def step_e2e():
        cond_mod.encoder = pinned_encoder
        try:
            wav = mg.generate(descriptions)            # the public API call (genmodel.py:151-171)
        finally:
            cond_mod.encoder = synth_enc
        return wav.to('cpu', non_blocking=False)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()

    def timed(fn, n):
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(n):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms, out

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    l0 = cm.launches
    with ClockSampler(torch.cuda.current_device()) as clk:
        ms, (tokens, wav) = timed(step_device, args.steps)
    clocks = clk.summary()
    dec_launches = (cm.launches - l0) // args.steps   # EnCodec decode kernels per generate
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(tokens=tokens, wav=wav))
    del tokens, wav
    audio_s = total_items * dur * args.steps
    value = audio_s / (ms / 1e3)
    n_e2e = max(1, min(args.steps, 3))
    ms_e2e, wav_host = timed(step_e2e, n_e2e)
    e2e_value = total_items * dur * n_e2e / (ms_e2e / 1e3)
    d2h_bytes = wav_host.numel() * 4

    # ---- dominant kernel, timed in isolation with CUDA events on the launching stream (acb_lm_debug_gemms enqueues only it).
    # Fused step: the dominant kernel IS the step (lm_step_kernel, one launch per decode step); its algorithmic bytes depend
    # on the KV length, so it is timed at 5 pinned lengths and the generation is integrated over them (trapezoid).
    # Per-phase path (ACB_LM_STEP=v5): lm_gemm_kernel, one pass = every weight matrix of a step.
    # Either way one launch / pass streams W_step = 3.2 GB >> 126 MB L2: no L2 reuse between timed launches.
    rows = 2 * B
    w_step, kv_tok, total_bytes = algorithmic_bytes(lm, rows, S)
    pk = peaks()
    nl = C.c_int(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fused = lm.launches_per_step <= 4

    def time_dominant(reps):
        for _ in range(3):
            _lib.check(lm._lib.acb_lm_debug_gemms(lm._handle, _lib.stream(), C.byref(nl)))
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            _lib.check(lm._lib.acb_lm_debug_gemms(lm._handle, _lib.stream(), C.byref(nl)))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    traffic = None
    step_ms = ms / args.steps / (S - 1)  # whole generate incl. sampler and EnCodec decode, amortised per decode step
    whole = dict(algorithmic_bytes=total_bytes, achieved=round(total_bytes / (ms / args.steps / 1e3) / 1e9, 1),
                 frac=round(total_bytes / (ms / args.steps / 1e3) / 1e9 / pk['hbm_gbs'], 4), ms_per_decode_step=round(step_ms, 4))
    if fused:
        pts = []
        for t in (0, (S - 2) // 4, (S - 2) // 2, 3 * (S - 2) // 4, S - 2):
            lm._bufs['pos'][0] = t
            k_ms = time_dominant(10)
            byt = w_step + rows * (t + 1) * kv_tok + rows * kv_tok
            pts.append(dict(kv_len=t + 1, ms=round(k_ms, 4), algorithmic_bytes=byt, gbs=round(byt / k_ms / 1e6, 1)))
        tot_ms = sum((pts[i]['ms'] + pts[i + 1]['ms']) / 2 * (pts[i + 1]['kv_len'] - pts[i]['kv_len']) for i in range(len(pts) - 1))
        mid = pts[len(pts) // 2]
        achieved = total_bytes / (tot_ms / 1e3) / 1e9
        tp = os.path.join(ROOT, 'profiles', 'r2_step_kernel_dram.json')   # ncu --set full capture of lm_step_kernel at KV 752
        if os.path.exists(tp) and args.scale == 'medium' and B == 8:
            tj = json.load(open(tp))
            traffic = int(tj['dram_bytes_read'] + tj['dram_bytes_write'])
        roofline = dict(bound='hbm', kernel='lm_step_kernel', achieved=round(achieved, 1), peak=pk['hbm_gbs'], unit='GB/s',
                        frac=round(achieved / pk['hbm_gbs'], 4), traffic=traffic, peak_source=pk['source'],
                        how='algorithmic bytes of the S-1 step launches of one generate / their kernel time, the latter integrated '
                            'from CUDA-event timings of the isolated kernel at the listed KV lengths; traffic = ncu dram bytes of the '
                            'launch at kv_len ' + str(mid['kv_len']) + ' (algorithmic ' + str(mid['algorithmic_bytes']) + ' B)',
                        launches_per_generate=S - 1, kernel_ms_per_generate=round(tot_ms, 2), per_kv=pts, whole_generate=whole)
    else:
        gemm_ms = time_dominant(20)
        tp = os.path.join(ROOT, 'profiles', 'r2_step_kv751_dram_summary.json')   # ncu launch list + DRAM bytes of the per-phase kernels (round 2)
        if os.path.exists(tp) and args.scale == 'medium' and B == 8:
            tj = json.load(open(tp)).get('lm_gemm_kernel')
            if tj:
                traffic = int((tj['dram_read_MB'] + tj['dram_write_MB']) * 1e6)
        achieved = w_step / (gemm_ms / 1e3) / 1e9
        roofline = dict(bound='hbm', kernel='lm_gemm_kernel', achieved=round(achieved, 1), peak=pk['hbm_gbs'], unit='GB/s',
                        frac=round(achieved / pk['hbm_gbs'], 4), traffic=traffic, peak_source=pk['source'],
                        launches_per_pass=nl.value, bytes_per_pass=w_step, ms_per_pass=round(gemm_ms, 4), whole_generate=whole)

    # ---- secondary metric: EnCodec 32 kHz encode+decode MSamples/s (BASELINE configs[3] per-GPU slice, 32 x 10 s)
    secondary = None
    if not args.no_encodec:
        xb = torch.randn(32, 1, 320000, device=dev) * 0.1
        for _ in range(2):
            c_, _s = cm.encode(xb)
            cm.decode(c_)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            c_, _s = cm.encode(xb)
            y_ = cm.decode(c_)
        e1.record()
        torch.cuda.synchronize()
        enc_ms = e0.elapsed_time(e1) / 3
        secondary = dict(metric='EnCodec 32kHz encode+decode MSamples/sec', value=round(xb.numel() / (enc_ms / 1e3) / 1e6, 2),
                         unit='MSamples/s', config='32 x 10 s mono per GPU; encoder fp32-accurate and index-exact (3xTF32 with bounded tensor-core accumulation runs: conv1d_t6 on tcgen05, fused residual blocks and the LSTM step on mma.sync; fp32 FMA where neither wins), decoder 3xTF32 (tcgen05 convolutions, fused residual blocks)',
                         ms=round(enc_ms, 2), roofline=encodec_roofline(xb.numel(), enc_ms))
        # throughput mode: the encoder's convolutions on the tensor cores as well (latents within 1.5e-4 of fp32)
        from audiocraft_b200 import synth as _synth
        from audiocraft_b200.encodec import EncodecModel as _EM
        _cfg = _synth.ENCODEC_CONFIGS['encodec_32k']
        cm_fast = _EM(_synth.synth_encodec_state_dict(_cfg, 1), _cfg, dev, encoder_precision='tf32x3')
        for _ in range(2):
            c_, _s = cm_fast.encode(xb)
            cm_fast.decode(c_)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            c_, _s = cm_fast.encode(xb)
            y_ = cm_fast.decode(c_)
        e1.record()
        torch.cuda.synchronize()
        fast_ms = e0.elapsed_time(e1) / 3
        secondary['tensor_core_encoder'] = dict(value=round(xb.numel() / (fast_ms / 1e3) / 1e6, 2), unit='MSamples/s', ms=round(fast_ms, 2))
        del cm_fast

    cpu_baseline = None
    reference_gpu = None
    if rank == 0 and args.gpus == 1 and not args.no_ref_gpu:
        # the reference's own CUDA path on this box (both models stay resident: ~15 GB of 180)
        from baseline import reference_arm as RA
        if RA.available():
            try:
                reference_gpu = RA.gpu_reference(args.scale, B, dur, passes=2, encodec_items=0 if args.no_encodec else 32)
            except Exception as ex:   # the arm must never take the product line down
                reference_gpu = dict(unavailable=f'{type(ex).__name__}: {ex}'[:300])
            torch.cuda.empty_cache()
        else:
            reference_gpu = dict(unavailable='baseline/_ref is not installed')
    if rank == 0 and args.gpus == 1 and not args.no_cpu:
        cpu_baseline = cpu_reference(args)
        if secondary is not None:
            from baseline import reference_arm as RA
            if RA.available():
                secondary['cpu_baseline'] = RA.cpu_encodec_baseline(1, 10.0)

    if rank == 0:
        line = dict(metric=METRIC, value=round(value, 2), unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=round(ms / args.steps, 2), higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                    dtype='f16', data='synthetic',
                    config=dict(workload=f'MusicGen-{args.scale} text-conditioned {dur:g}s generation, batch={B} per GPU '
                                         f'(CFG rows={2 * B}), top_k=250, EnCodec-32k decode included',
                                global_batch=total_items, seq_len=T,
                                parallelism=(f'dp{world}: one batch of {args.batch} split over the ranks, waveforms all-gathered (NCCL) in the timed region'
                                             if strong else f'dp{world} (batch split, no collective)'),
                                limiter=('per-replica weight stream: every rank re-reads the %.2f GB of weights per decode step at the same '
                                         'latency-bound step time whatever its share of the batch' % (w_step / 1e9)) if strong else None,
                                pdl=bool(lm._lib.acb_lm_uses_pdl(lm._handle)),
                                l2='inputs larger than L2: every decode step streams %.2f GB of weights' % (w_step / 1e9)),
                    clocks=clocks,
                    e2e=dict(value=round(e2e_value, 2), unit=UNIT, h2d_bytes_per_step=h2d_bytes, d2h_bytes_per_step=d2h_bytes),
                    gpu_launches=(lm.launches_per_step * (S - 1) + dec_launches) * args.steps,
                    roofline=roofline, cpu_baseline=cpu_baseline, reference_gpu=reference_gpu, secondary=secondary)
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def cpu_reference(args, n_samples=2):
    """cpu_baseline: the reference's own modules (baseline/_ref) on the host cores, bounded samples (reference_arm.py)."""
    from baseline import reference_arm as RA
    if not RA.available():
        return dict(value=None, unit=UNIT, cores=0, kind='unavailable', sample='baseline/_ref is not installed (baseline/install_ref.sh)')
    return RA.cpu_baseline(args.scale, args.batch, args.duration, n_samples=n_samples, n_steps=args.cpu_steps)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from baseline import reference_arm as RA
    if not RA.available():
        emit(dict(impl='reference', unavailable='baseline/_ref is not installed (run baseline/install_ref.sh in the build container)'))
        return
    from oracle import ref_import as R
    ref = RA.CpuReference(args.scale, args.batch, args.duration)
    for _ in range(args.warmup):
        ref.sample(n_steps=1, ctx=64)
    smps = [ref.sample(n_steps=args.cpu_steps) for _ in range(args.steps)]
    order = sorted(smps, key=lambda q: q['value'])
    med = order[len(order) // 2]
    cb = dict(value=round(med['value'], 4), unit=UNIT, cores=ref.threads, kind='reference' if R.kind() == '_ref' else 'reference-tree',
              sample=ref.describe(med), spread=[round(q['value'], 4) for q in smps])
    line = dict(metric=METRIC, value=cb['value'], unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=round(sum(q['wall_s'] for q in smps) / len(smps) * 1e3, 1), higher_is_better=True, scaling='weak',
                vs_baseline=None, dtype='f32', data='synthetic', impl='reference',
                config=dict(workload=f'MusicGen-{args.scale} text-conditioned {args.duration:g}s generation, batch={args.batch} '
                                     f'(CFG rows={2 * args.batch}), top_k=250, EnCodec-32k decode included; each step is a bounded '
                                     f'sample integrated to the full pass (cpu_baseline.sample)',
                            global_batch=args.batch, seq_len=int(args.duration * 50), parallelism='host cores (rank 0 only)'),
                gpu_launches=0, cpu_baseline=cb,
                e2e=dict(value=cb['value'], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    emit(line)


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line to stdout when
    the box sets NCCL_DEBUG): keep a private handle on the real stdout for the result and point fd 1 at stderr for
    everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


if __name__ == '__main__':
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--scale', default='medium', choices=['small', 'medium', 'large'])
    ap.add_argument('--duration', type=float, default=30.0)
    ap.add_argument('--batch', type=int, default=8)
    ap.add_argument('--cpu-steps', type=int, default=4, help='decode steps per KV window of one CPU reference sample')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'])
    ap.add_argument('--workload', default='musicgen', choices=['musicgen', 'encodec'])
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-ref-gpu', action='store_true', help='skip timing the reference CUDA path (reference_gpu block)')
    ap.add_argument('--no-encodec', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs applies to --impl b200')
    if a.impl == 'reference':
        run_reference(a)
    elif a.workload == 'encodec':
        run_encodec(a)
    else:
        run_b200(a)
