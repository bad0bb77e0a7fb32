"""HiFi-GAN(-NSF) vocoder plugin backed by libsvb_vocoder.so.

Same surface as the reference class (vocoders/hifigan.py:39-69 + PWG.wav2spec,
vocoders/pwg.py:105-122): no-arg constructor reading ``hparams['vocoder_ckpt']``,
``spec2wav(mel[T,80], f0=[T]) -> np.float32[T*hop]``, static ``wav2spec(wav_fn)``,
registered under the names ``HifiGAN`` / ``hifigan``.
"""
import ctypes
import glob
import json
import os
import re

import numpy as np
import torch

from neuralsvb_b200 import _native, utils
from neuralsvb_b200.modules.hifigan.hifigan import HifiGanGenerator
from neuralsvb_b200.utils import audio
from neuralsvb_b200.utils.hparams import hparams, set_hparams
from neuralsvb_b200.vocoders.base_vocoder import BaseVocoder, register_vocoder


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('neuralsvb_b200.vocoders.hifigan needs a CUDA device: the B200 path has no CPU fallback')
    return torch.device('cuda', torch.cuda.current_device())


def load_model(config_path, checkpoint_path):
    """reference: vocoders/hifigan.py:17-33 (yaml -> ckpt['state_dict']['model_gen'],
    json -> ckpt['generator']; strict load; fold weight norm; eval on the GPU)."""
    device = _require_cuda()
    ckpt_dict = torch.load(checkpoint_path, map_location='cpu', weights_only=False)
    if '.yaml' in config_path:
        config = set_hparams(config_path, global_hparams=False)
        state = ckpt_dict['state_dict']['model_gen']
    elif '.json' in config_path:
        with open(config_path) as f:
            config = json.load(f)
        state = ckpt_dict['generator']
    else:
        raise ValueError(f'unknown vocoder config type: {config_path}')
    model = HifiGanGenerator(config)
    model.load_state_dict(state, strict=True)
    model.remove_weight_norm()
    model = model.eval().to(device)
    model.native_handle(device)                     # pack + upload once, like .to(device)
    print(f'| Loaded model parameters from {checkpoint_path}.')
    print(f'| HifiGAN device: {device}.')
    return model, config, device


def stft_config(hp, pad_mode, out_kind, eps, frames_major=1, clamp=0):
    c = _native.StftConfig()
    c.n_fft, c.hop, c.win = int(hp['fft_size']), int(hp['hop_size']), int(hp['win_size'])
    c.pad_mode, c.out_kind, c.clamp_input = pad_mode, out_kind, clamp
    c.n_mels, c.frames_major, c.eps = int(hp['audio_num_mel_bins']), frames_major, float(eps)
    return c


def _load_wav(wav_fn, sr):
    from scipy.io import wavfile
    file_sr, data = wavfile.read(wav_fn)
    if data.dtype.kind == 'i':
        data = data.astype(np.float32) / float(np.iinfo(data.dtype).max + 1)
    elif data.dtype.kind == 'u':
        data = (data.astype(np.float32) - 128.0) / 128.0
    data = data.astype(np.float32)
    if data.ndim > 1:
        data = data.mean(axis=1)
    if file_sr != sr:
        raise ValueError(f'{wav_fn}: sample rate {file_sr} != audio_sample_rate {sr}; resampling '
                         '(librosa.core.load in the reference) is data preparation, outside this path')
    return data


@register_vocoder
class HifiGAN(BaseVocoder):
    def __init__(self):
        base_dir = hparams['vocoder_ckpt']
        config_path = f'{base_dir}/config.yaml'
        if os.path.exists(config_path):
            ckpts = glob.glob(f'{base_dir}/model_ckpt_steps_*.ckpt')
            ckpt = sorted(ckpts, key=lambda x: int(re.findall(r'model_ckpt_steps_(\d+)\.ckpt', x)[0]))[-1]
            print('| load HifiGAN: ', ckpt)
            self.model, self.config, self.device = load_model(config_path=config_path, checkpoint_path=ckpt)
        else:
            config_path = f'{base_dir}/config.json'
            ckpt = f'{base_dir}/generator_v1'
            if os.path.exists(config_path):
                self.model, self.config, self.device = load_model(config_path=config_path, checkpoint_path=ckpt)
            else:
                raise FileNotFoundError(f'no config.yaml / config.json under vocoder_ckpt={base_dir!r}')

    @classmethod
    def from_model(cls, model, config, device=None):
        """Build the plugin around an in-memory generator (no checkpoint directory)."""
        self = cls.__new__(cls)
        self.device = device or _require_cuda()
        self.model, self.config = model.eval().to(self.device), config
        self.model.native_handle(self.device)
        return self

    def spec2wav(self, mel, **kwargs):
        """mel [T, n_mel] (numpy or CPU tensor, log10-mel), f0=[T] Hz or None -> np.float32 [T*hop]."""
        return self.spec2wav_batch(np.asarray(mel, dtype=np.float32)[None],
                                   None if kwargs.get('f0') is None
                                   else np.asarray(kwargs['f0'], dtype=np.float32)[None],
                                   seed=kwargs.get('seed'))[0]

    def spec2wav_batch(self, mels, f0s=None, seed=None, int16=False, norm=False):
        """mels [B, T, n_mel], f0s [B, T] or None (host arrays) -> np.float32 [B, T*hop].
        One call = pinned staging + H2D + generator + D2H + stream sync (svb_gen_spec2wav_host).
        ``int16=True``: save_wav's sample conversion (utils/audio.py:11-16; ``norm`` = its peak normalisation) runs on
        the device and np.int16 [B, T*hop] comes back -- half the D2H bytes, nothing left for the CPU writer pool to do
        but ``wavfile.write`` (svb_gen_spec2wav_host_i16; the denoise post-filter needs the float path)."""
        mels = np.ascontiguousarray(mels, dtype=np.float32)
        B, T, C = mels.shape
        if f0s is not None:
            f0s = np.ascontiguousarray(f0s, dtype=np.float32)
            assert f0s.shape == (B, T), (f0s.shape, (B, T))
        lib = _native.lib()
        g = self.model.native_handle(self.device)
        hop = int(lib.svb_gen_hop(g))
        if int16 and hparams.get('vocoder_denoise_c', 0.0) > 0:
            raise ValueError('int16 output and vocoder_denoise_c > 0 are exclusive (the post-filter works on floats)')
        out = np.empty((B, T * hop), np.int16 if int16 else np.float32)
        if seed is None:
            self.model.seed += 1
            seed = self.model.seed
        if int16:
            with torch.no_grad(), torch.cuda.device(self.device):
                with utils.Timer('hifigan', enable=hparams.get('profile_infer', False)):
                    _native.check(lib.svb_gen_spec2wav_host_i16(
                        g, mels.ctypes.data_as(ctypes.c_void_p),
                        None if f0s is None else f0s.ctypes.data_as(ctypes.c_void_p),
                        ctypes.c_uint64(seed), B, T, int(bool(norm)), out.ctypes.data_as(ctypes.c_void_p),
                        _native.current_stream_ptr(self.device)), 'spec2wav_i16')
            return out
        with torch.no_grad(), torch.cuda.device(self.device):
            with utils.Timer('hifigan', enable=hparams.get('profile_infer', False)):
                st = _native.current_stream_ptr(self.device)
                _native.check(lib.svb_gen_spec2wav_host(
                    g, mels.ctypes.data_as(ctypes.c_void_p),
                    None if f0s is None else f0s.ctypes.data_as(ctypes.c_void_p),
                    ctypes.c_uint64(seed), B, T, out.ctypes.data_as(ctypes.c_void_p), st), 'spec2wav')
        if hparams.get('vocoder_denoise_c', 0.0) > 0:                  # vocoders/hifigan.py:66-69
            from neuralsvb_b200.vocoders.vocoder_utils import denoise
            out = np.stack([denoise(o, v=hparams['vocoder_denoise_c']) for o in out])
        return out

    def spec2wav_ragged(self, mels, f0s=None, seed=None, int16=False, norm=False):
        """Clips of different lengths in one call: list of mel [T_b, n_mel] (host arrays), f0s list of [T_b] or None ->
        list of np.float32 [T_b*hop] (np.int16 with ``int16=True``).  One H2D of the packed clips, one ragged generator
        forward, one D2H (svb_gen_spec2wav_ragged_host[_i16]); clip b equals ``forward(..., lengths=...)`` on the padded batch.
        The float path applies ``denoise`` per clip when ``vocoder_denoise_c > 0``; ``norm`` takes each clip's own peak."""
        mels = [np.ascontiguousarray(m, dtype=np.float32) for m in mels]
        if not mels:
            return []
        lens = np.array([m.shape[0] for m in mels], np.int32)
        if any(m.ndim != 2 or m.shape[1] != mels[0].shape[1] for m in mels):
            raise ValueError('every mel must be [T_b, n_mel] with the same n_mel')
        cat = np.ascontiguousarray(np.concatenate(mels))
        f0cat = None
        if f0s is not None:
            f0s = [np.asarray(f, dtype=np.float32).reshape(-1) for f in f0s]
            if [len(f) for f in f0s] != lens.tolist():
                raise ValueError('f0s must have one [T_b] array per mel')
            f0cat = np.ascontiguousarray(np.concatenate(f0s))
        lib = _native.lib()
        g = self.model.native_handle(self.device)
        hop = int(lib.svb_gen_hop(g))
        if int16 and hparams.get('vocoder_denoise_c', 0.0) > 0:
            raise ValueError('int16 output and vocoder_denoise_c > 0 are exclusive (the post-filter works on floats)')
        out = np.empty(int(lens.sum()) * hop, np.int16 if int16 else np.float32)
        if seed is None:
            self.model.seed += 1
            seed = self.model.seed
        vp = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
        with torch.no_grad(), torch.cuda.device(self.device):
            with utils.Timer('hifigan', enable=hparams.get('profile_infer', False)):
                st = _native.current_stream_ptr(self.device)
                if int16:
                    _native.check(lib.svb_gen_spec2wav_ragged_host_i16(g, vp(cat), vp(f0cat), vp(lens), len(mels), ctypes.c_uint64(seed),
                                                                       int(bool(norm)), vp(out), st), 'spec2wav_ragged_i16')
                else:
                    _native.check(lib.svb_gen_spec2wav_ragged_host(g, vp(cat), vp(f0cat), vp(lens), len(mels), ctypes.c_uint64(seed),
                                                                   vp(out), st), 'spec2wav_ragged')
        wavs = np.split(out, np.cumsum(lens.astype(np.int64) * hop)[:-1])
        if not int16 and hparams.get('vocoder_denoise_c', 0.0) > 0:       # vocoders/hifigan.py:66-69, per clip
            from neuralsvb_b200.vocoders.vocoder_utils import denoise
            wavs = [denoise(w, v=hparams['vocoder_denoise_c']) for w in wavs]
        return wavs

    @staticmethod
    def wav2spec_batch(wav_fns, hp=None):
        """The binarizer's per-file ``wav2spec`` loop (data_gen/tts/base_binarizer.py:168-178,
        data_gen/singing/binarize_para.py:116-217) as ONE device call over a ragged batch: list of paths / float arrays
        -> list of (wav [T*hop], mel [T, n_mel] log10), identical to ``wav2spec`` clip by clip
        (svb_wav2spec_batch_host: one H2D, one launch over all frames of all clips, one D2H)."""
        hp = hparams if hp is None else hp
        device = _require_cuda()
        if hp.get('loud_norm', False):
            raise NotImplementedError('loud_norm (pyloudnorm BS.1770) is data preparation, outside this path')
        wavs = [_load_wav(w, hp['audio_sample_rate']) if isinstance(w, str) else np.ascontiguousarray(w, dtype=np.float32)
                for w in wav_fns]
        if not wavs:
            return []
        lib = _native.lib()
        cfg = stft_config(hp, _native.PAD_CENTER_ZERO, _native.OUT_LOG10_MEL, float(hp.get('wav2spec_eps', 1e-10)))
        lengths = np.array([len(w) for w in wavs], np.int64)
        frames = lengths // cfg.hop + 1
        cat = np.ascontiguousarray(np.concatenate(wavs))
        basis = np.ascontiguousarray(audio.build_mel_basis(hp))
        mel = np.empty((int(frames.sum()), cfg.n_mels), np.float32)
        got = np.zeros(len(wavs), np.int64)
        with torch.cuda.device(device):
            rc = lib.svb_wav2spec_batch_host(ctypes.byref(cfg), cat.ctypes.data_as(ctypes.c_void_p),
                                             lengths.ctypes.data_as(ctypes.c_void_p), len(wavs),
                                             basis.ctypes.data_as(ctypes.c_void_p), mel.ctypes.data_as(ctypes.c_void_p),
                                             got.ctypes.data_as(ctypes.c_void_p), device.index,
                                             _native.current_stream_ptr(device))
            _native.check(rc, 'wav2spec_batch')
        assert np.array_equal(got, frames), (got, frames)
        out, o = [], 0
        for w, fr in zip(wavs, frames):
            n_out = int(fr) * cfg.hop                       # audio.librosa_pad_lr + wav[:T * hop] (data_gen_utils.py:138-140)
            wo = np.zeros(n_out, np.float32)
            wo[:min(len(w), n_out)] = w[:n_out]
            out.append((wo, mel[o:o + int(fr)]))
            o += int(fr)
        return out

    @staticmethod
    def wav2spec(wav_fn, return_linear=False, hp=None):
        """wav file path (same sample rate) or float array -> (wav [T*hop], mel [T, n_mel] log10)
        [+ normalised dB linear spectrogram [T, n_fft/2+1]]   (vocoders/pwg.py:105-122)."""
        hp = hparams if hp is None else hp
        device = _require_cuda()
        if hp.get('loud_norm', False):
            raise NotImplementedError('loud_norm (pyloudnorm BS.1770) is data preparation, outside this path')
        wav = _load_wav(wav_fn, hp['audio_sample_rate']) if isinstance(wav_fn, str) \
            else np.ascontiguousarray(wav_fn, dtype=np.float32)
        eps = float(hp.get('wav2spec_eps', 1e-10))
        lib = _native.lib()
        cfg = stft_config(hp, _native.PAD_CENTER_ZERO, _native.OUT_LOG10_MEL, eps)
        frames = int(lib.svb_stft_num_frames(ctypes.byref(cfg), len(wav)))
        basis = np.ascontiguousarray(audio.build_mel_basis(hp))
        mel = np.empty((frames, cfg.n_mels), np.float32)
        wav_out = np.empty(frames * cfg.hop, np.float32)
        with torch.cuda.device(device):
            st = _native.current_stream_ptr(device)
            rc = lib.svb_wav2spec_host(ctypes.byref(cfg), wav.ctypes.data_as(ctypes.c_void_p), len(wav),
                                       basis.ctypes.data_as(ctypes.c_void_p), mel.ctypes.data_as(ctypes.c_void_p),
                                       wav_out.ctypes.data_as(ctypes.c_void_p), device.index, st)
            _native.check(rc, 'wav2spec')
            if not return_linear:
                return wav_out, mel
            cfg2 = stft_config(hp, _native.PAD_CENTER_ZERO, _native.OUT_MAG_RAW, 0.0)
            w = torch.from_numpy(wav).to(device)
            lin = torch.empty(frames, cfg.n_fft // 2 + 1, device=device)
            _native.check(lib.svb_stft_forward(ctypes.byref(cfg2), _native.ptr(w), 1, len(wav), None,
                                               _native.ptr(lin), st), 'stft_forward')
            lin = audio.normalize(audio.amp_to_db(lin.cpu().numpy()), hp)
        return wav_out, mel, lin
