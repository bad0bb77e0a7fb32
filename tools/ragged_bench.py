"""Ragged batches through the HiFi-GAN-NSF generator: one forward(lengths=...) against the alternatives a user has without it.

Full hop-256 NSF config (S.hifigan_config) in bf16x3, Philox noise, inputs resident in HBM, CUDA events around every call.
Every shape is warmed up first; the arms alternate inside each repetition and the median of --reps repetitions is reported.
Rates are audio-seconds per second of VALID audio (sum of the clips' lengths), whatever the arm computes.

  A: 16 clips of np.random.RandomState(1234).randint(86, 1379, 16) frames (1-16 s at 22.05 kHz)
     1 ragged   forward(lengths=...) in one call
     2 loop     one B = 1 forward per clip
     3 padded   plain forward of the batch padded to the longest clip (NOT equivalent: the tails differ)
  B: 16 x 688 frames (equal lengths)
     4 uniform  svb_gen_forward  vs  ragged  svb_gen_forward_ragged with every length 688 (overhead of the ragged path)
  5 (A, end to end from host memory): HifiGAN.spec2wav_ragged vs a loop of HifiGAN.spec2wav

    python tools/ragged_bench.py [--reps 20] [--out profiles/r03_ragged_bench.json]
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neuralsvb_b200.modules.hifigan.hifigan import HifiGanGenerator  # noqa: E402
from neuralsvb_b200.utils import synthetic as S  # noqa: E402


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return {'device': name, 'power_limit_and_max_sm_clock': q}


def timed(fn):
    """ms of fn() between CUDA events on the current stream (fn may synchronise the host itself)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default='profiles/r03_ragged_bench.json')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('ragged_bench needs a CUDA device: there is nothing to measure on the CPU')
    torch.cuda.set_device(0)
    info = device_info()
    print(info)

    h = S.hifigan_config()
    hop, sr = 256, h['audio_sample_rate']
    m = HifiGanGenerator(h, precision='bf16x3')
    m.load_state_dict(S.make_generator_state_dict(h, 1234), strict=True)
    with contextlib.redirect_stdout(io.StringIO()):
        m.remove_weight_norm()
    m = m.eval().cuda()

    lens_a = np.random.RandomState(1234).randint(86, 1379, 16).tolist()
    Ta = max(lens_a)
    mel_a, f0_a = S.make_mel_f0(16, Ta, 1234)
    mel_a, f0_a = mel_a.cuda(), f0_a.cuda()
    clips = [(mel_a[b:b + 1, :, :L].contiguous(), f0_a[b:b + 1, :L].contiguous()) for b, L in enumerate(lens_a)]
    Tb = 688
    mel_b, f0_b = S.make_mel_f0(16, Tb, 4321)
    mel_b, f0_b = mel_b.cuda(), f0_b.cuda()
    lens_b = [Tb] * 16

    from neuralsvb_b200.vocoders.hifigan import HifiGAN
    from neuralsvb_b200.utils.hparams import hparams
    hparams['vocoder_denoise_c'] = 0.0
    voc = HifiGAN.from_model(m, h)
    mels_host = [mel_a[b, :, :L].T.contiguous().cpu().numpy() for b, L in enumerate(lens_a)]
    f0s_host = [f0_a[b, :L].cpu().numpy() for b, L in enumerate(lens_a)]

    def loop():
        for mc, fc in clips:
            m(mc, fc, seed=1)

    def loop_host():
        for mh, fh in zip(mels_host, f0s_host):
            voc.spec2wav(mh, f0=fh, seed=1)

    arms = {
        'A1_ragged_one_call': (lambda: m(mel_a, f0_a, seed=1, lengths=lens_a), lens_a),
        'A2_loop_of_B1': (loop, lens_a),
        'A3_padded_not_equivalent': (lambda: m(mel_a, f0_a, seed=1), lens_a),
        'B4_uniform_svb_gen_forward': (lambda: m(mel_b, f0_b, seed=1), lens_b),
        'B4_uniform_svb_gen_forward_ragged': (lambda: m(mel_b, f0_b, seed=1, lengths=lens_b), lens_b),
        'A5_spec2wav_ragged_host': (lambda: voc.spec2wav_ragged(mels_host, f0s_host, seed=1), lens_a),
        'A5_loop_of_spec2wav_host': (loop_host, lens_a),
    }
    # the equivalence the speed comparison rests on: arm 1 and arm 2 compute the same samples
    with torch.no_grad():
        ri, nz = S.make_nsf_noise(16, Ta * hop, 1234)
        ri, nz = ri.cuda(), nz.cuda()
        yr = m(mel_a, f0_a, rand_ini=ri, noise=nz, lengths=lens_a)
        same = all(torch.equal(yr[b:b + 1, :, :L * hop],
                               m(clips[b][0], clips[b][1], rand_ini=ri[b:b + 1].contiguous(), noise=nz[b:b + 1, :L * hop].contiguous()))
                   for b, L in enumerate(lens_a))
    del yr, ri, nz
    print(f'arm 1 == arm 2 clip by clip (injected noise, bitwise): {same}')

    times = {k: [] for k in arms}
    with torch.no_grad():
        for _ in range(args.warmup):
            for k, (fn, _) in arms.items():
                timed(fn)
        t_start = time.time()
        for r in range(args.reps):
            for k, (fn, _) in arms.items():                  # alternate the arms inside every repetition
                times[k].append(timed(fn))
        wall = time.time() - t_start
    res = {}
    for k, (_, lens) in arms.items():
        ms = float(np.median(times[k]))
        audio_s = sum(lens) * hop / sr
        res[k] = {'median_ms': round(ms, 3), 'min_ms': round(float(np.min(times[k])), 3), 'max_ms': round(float(np.max(times[k])), 3),
                  'valid_audio_s': round(audio_s, 3), 'valid_audio_s_per_s': round(audio_s / (ms / 1e3), 1)}
        print(f'{k:36s} median {ms:9.3f} ms  [{np.min(times[k]):.3f} .. {np.max(times[k]):.3f}]  {audio_s / (ms / 1e3):10.1f} audio-s/s')
    out = {'what': 'tools/ragged_bench.py: HiFi-GAN-NSF hop-256 bf16x3 generator, ragged vs per-clip vs padded', **info,
           'reps': args.reps, 'warmup': args.warmup, 'timed_window_s': round(wall, 1),
           'workload_A_frames': lens_a, 'workload_B_frames': lens_b, 'arm1_equals_arm2_bitwise': bool(same), 'arms': res,
           'ratios': {'A1_vs_A2_speedup': round(res['A2_loop_of_B1']['median_ms'] / res['A1_ragged_one_call']['median_ms'], 3),
                      'A1_vs_A3_speedup': round(res['A3_padded_not_equivalent']['median_ms'] / res['A1_ragged_one_call']['median_ms'], 3),
                      'B4_ragged_over_uniform_time': round(res['B4_uniform_svb_gen_forward_ragged']['median_ms'] /
                                                           res['B4_uniform_svb_gen_forward']['median_ms'], 4),
                      'A5_host_speedup': round(res['A5_loop_of_spec2wav_host']['median_ms'] / res['A5_spec2wav_ragged_host']['median_ms'], 3)}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out['ratios']))


if __name__ == '__main__':
    main()
