"""ORACLE tooling (test infrastructure only; see oracle/__init__.py).

Writes tests/golden/*.npz from the UNMODIFIED reference modules under
/root/reference (via oracle/ref_harness.py).  Build container only; the
fixtures are committed so the GPU box (no /root/reference) can still check the
oracle and the CUDA path against reference outputs.

    python -m oracle.gen_golden            # regenerate everything

Inputs and weights are never stored: they are regenerated bit-identically by
neuralsvb_b200/utils/synthetic.py from the seeds recorded in each fixture.
"""
import os
import sys
import warnings

import numpy as np
import torch

from neuralsvb_b200.utils import synthetic as S
from oracle import ref_harness as R

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
SEED = 1234

FRONTEND_CASES = {
    # name: (n_samples, fft, hop, win, fmin, fmax)      SURVEY 8(d) cfg 1 + D6 variants
    'cfg1_win512': (44100, 1024, 256, 512, 80, 7600),
    'cfg1_win1024': (22050, 1024, 256, 1024, 80, 7600),
    'svb_hop128': (22050, 512, 128, 512, 50, 11025),
    'ragged_short': (1000, 1024, 256, 512, 80, 7600),
}


def gen_frontend():
    R.install()
    from data_gen.tts.data_gen_utils import process_utterance        # the real reference function
    out = {}
    for name, (n, fft, hop, win, fmin, fmax) in FRONTEND_CASES.items():
        wav = S.make_clip(n, seed=SEED)
        w2, mel, lin = process_utterance(wav, fft_size=fft, hop_size=hop, win_length=win, num_mels=80,
                                         fmin=fmin, fmax=fmax, sample_rate=22050, eps=1e-10,
                                         return_linear=True, min_level_db=-100)
        out[f'{name}/mel'] = mel.T.astype(np.float32)                # [T, 80] as PWG.wav2spec returns it
        out[f'{name}/wav_len'] = np.int64(len(w2))
        out[f'{name}/lin_sub'] = lin.T[::7, ::5].astype(np.float32)
        out[f'{name}/params'] = np.array([n, fft, hop, win, fmin, fmax], np.int64)
    np.savez_compressed(os.path.join(OUT, 'frontend.npz'), **out)
    print('frontend.npz', {k: v.shape for k, v in out.items() if k.endswith('/mel')})


GEN_CASES = {
    # name: (config, B, T_frames, nsf, subsample stride)
    'small_nsf': ('small', 2, 24, True, 1),
    'small_plain': ('small', 2, 24, False, 1),
    'small_ragged': ('small', 1, 37, True, 1),
    'hop256_t16': ('hop256', 1, 16, True, 1),
    'hop256_t21_plain': ('hop256', 1, 21, False, 1),
    'cfg2_b16_t128': ('hop256', 16, 128, True, 61),
}


def _cfg(name, nsf):
    return S.small_config(nsf) if name == 'small' else S.hifigan_config(nsf)


def gen_generator():
    out = {}
    for name, (cfg, B, T, nsf, stride) in GEN_CASES.items():
        h = _cfg(cfg, nsf)
        hop = int(np.prod(h['upsample_rates']))
        sd = S.make_generator_state_dict(h, SEED)
        mel, f0 = S.make_mel_f0(B, T, SEED)
        model = R.build_generator(h, sd)
        if nsf:
            ri, nz = S.make_nsf_noise(B, T * hop, SEED)
            y = R.run_generator(model, mel, f0, ri, nz)
            with R.injected_noise(ri, nz), torch.no_grad():
                f0_up = model.f0_upsamp(f0[:, None]).transpose(1, 2)
                har, _, _ = model.m_source(f0_up)
            out[f'{name}/har_sub'] = har[:, :, 0].numpy()[:, ::stride].astype(np.float32)
        else:
            y = R.run_generator(model, mel, None)
        y = y.numpy()[:, 0]
        out[f'{name}/y_sub'] = y[:, ::stride].astype(np.float32)
        out[f'{name}/rms'] = np.sqrt((y.astype(np.float64) ** 2).mean(axis=1))
        out[f'{name}/meta'] = np.array([B, T, int(nsf), stride, hop], np.int64)
        print(name, y.shape, 'rms', out[f'{name}/rms'].mean())
    np.savez_compressed(os.path.join(OUT, 'generator.npz'), **out)


def gen_losses():
    R.install()
    from modules.hifigan.mel_utils import mel_spectrogram
    from modules.parallel_wavegan.losses.stft_loss import MultiResolutionSTFTLoss, stft
    out = {}
    h = S.hifigan_config()
    y = S.make_wave_batch(2, 8192, seed=SEED)
    x = (y + 0.05 * S.make_wave_batch(2, 8192, seed=SEED + 1)).clamp(-1, 1)
    with R.legacy_stft(), torch.no_grad():
        out['mel_spectrogram/y'] = mel_spectrogram(y, h).numpy().astype(np.float32)          # [2, 80, 32]
        sc, mag = MultiResolutionSTFTLoss()(x, y)
        out['mr_stft/sc_mag'] = np.array([float(sc), float(mag)], np.float64)
        for fs, ss, wl in ((1024, 120, 600), (2048, 240, 1200), (512, 50, 240)):
            m = stft(x, fs, ss, wl, torch.hann_window(wl))
            out[f'stft_mag/{fs}'] = m.numpy()[:, ::3, ::7].astype(np.float32)
            out[f'stft_mag/{fs}_shape'] = np.array(m.shape, np.int64)
    np.savez_compressed(os.path.join(OUT, 'losses.npz'), **out)
    print('losses.npz', out['mr_stft/sc_mag'])


def gen_discriminators():
    """MPD / MSD (eval mode: spectral norm without power iteration) + GAN losses from the reference modules."""
    R.install()
    from utils.hparams import hparams as ref_hp
    ref_hp['hop_size'] = 256                                   # MultiScaleDiscriminator reads it at construction (:292-301)
    from modules.hifigan.hifigan import (MultiPeriodDiscriminator, MultiScaleDiscriminator, discriminator_loss, feature_loss,
                                         generator_loss)
    out = {}
    y = S.make_wave_batch(2, 8192, seed=SEED)[:, None]
    y_hat = (y + 0.1 * S.make_wave_batch(2, 8192, seed=SEED + 5)[:, None]).clamp(-1, 1)
    for name, cls, sd in (('mpd', MultiPeriodDiscriminator, S.make_mpd_state_dict(SEED)),
                          ('msd', MultiScaleDiscriminator, S.make_msd_state_dict(SEED))):
        m = cls()
        m.load_state_dict(sd, strict=True)
        m.eval()
        with torch.no_grad():
            rs, gs, fr, fg = m(y, y_hat)
            out[f'{name}/losses'] = np.array([float(feature_loss(fr, fg)), *[float(v) for v in discriminator_loss(rs, gs)],
                                              float(generator_loss(gs))], np.float64)
        for i, (r, g) in enumerate(zip(rs, gs)):
            out[f'{name}/logit_r{i}'], out[f'{name}/logit_g{i}'] = r.numpy(), g.numpy()
            for j, f in enumerate(fr[i]):
                out[f'{name}/fmap_r{i}_{j}_shape'] = np.array(f.shape, np.int64)
                out[f'{name}/fmap_r{i}_{j}_sub'] = f.numpy().reshape(-1)[::211].astype(np.float32)
        print(name, out[f'{name}/losses'])
    np.savez_compressed(os.path.join(OUT, 'discriminators.npz'), **out)


def gen_discriminators_cond():
    """use_cond=True variants (mel-conditioned cond_net, hifigan.py:185-189,204-206,257-260,274-276) from the reference
    modules: logits and the GAN losses."""
    R.install()
    from utils.hparams import hparams as ref_hp
    ref_hp['hop_size'] = 256
    from modules.hifigan.hifigan import (MultiPeriodDiscriminator, MultiScaleDiscriminator, cond_discriminator_loss,
                                         discriminator_loss, feature_loss, generator_loss)
    out = {}
    y = S.make_wave_batch(2, 8192, seed=SEED)[:, None]
    y_hat = (y + 0.1 * S.make_wave_batch(2, 8192, seed=SEED + 5)[:, None]).clamp(-1, 1)
    mel, _ = S.make_mel_f0(2, 32, SEED)
    for name, cls, sd in (('mpd', MultiPeriodDiscriminator, S.make_mpd_state_dict(SEED, use_cond=True)),
                          ('msd', MultiScaleDiscriminator, S.make_msd_state_dict(SEED, use_cond=True))):
        m = cls(use_cond=True)
        m.load_state_dict(sd, strict=True)
        m.eval()
        with torch.no_grad():
            rs, gs, fr, fg = m(y, y_hat, mel)
            out[f'{name}/losses'] = np.array([float(feature_loss(fr, fg)), *[float(v) for v in discriminator_loss(rs, gs)],
                                              float(generator_loss(gs)), float(cond_discriminator_loss(gs))], np.float64)
        for i, (r, g) in enumerate(zip(rs, gs)):
            out[f'{name}/logit_r{i}'], out[f'{name}/logit_g{i}'] = r.numpy(), g.numpy()
        print(name, out[f'{name}/losses'])
    np.savez_compressed(os.path.join(OUT, 'discriminators_cond.npz'), **out)


# ---------------------------------------------------------------------------------- round 2: branches the first set left unpinned
def extra_config(name, nsf=True):
    """Architectures of the extra generator cases (shared with the tests)."""
    if name == 'small_rb2':
        h = S.small_config(nsf)
        h['resblock'], h['resblock_dilation_sizes'] = '2', [[1, 3], [1, 3], [1, 3]]
    elif name == 'hop256_rb2':
        h = S.hifigan_config(nsf)
        h['resblock'], h['resblock_dilation_sizes'] = '2', [[1, 3], [1, 3], [1, 3]]
    elif name == 'hop128':
        h = S.hifigan_config(nsf, hop=128)
    else:
        raise KeyError(name)
    return h


GEN_EXTRA_CASES = {
    # name: (config, B, T_frames, nsf, subsample stride)      ResBlock2 (hifigan.py:70-91) and the hop-128 singing architecture
    'small_rb2': ('small_rb2', 2, 24, True, 1),
    'small_rb2_plain': ('small_rb2', 1, 37, False, 1),
    'hop256_rb2_t12': ('hop256_rb2', 1, 12, True, 1),
    'hop128_t20': ('hop128', 2, 20, True, 1),
}


def gen_generator_extra():
    out = {}
    for name, (cfg, B, T, nsf, stride) in GEN_EXTRA_CASES.items():
        h = extra_config(cfg, nsf)
        hop = int(np.prod(h['upsample_rates']))
        sd = S.make_generator_state_dict(h, SEED)
        mel, f0 = S.make_mel_f0(B, T, SEED)
        model = R.build_generator(h, sd)
        if nsf:
            ri, nz = S.make_nsf_noise(B, T * hop, SEED)
            y = R.run_generator(model, mel, f0, ri, nz)
        else:
            y = R.run_generator(model, mel, None)
        y = y.numpy()[:, 0]
        out[f'{name}/y_sub'] = y[:, ::stride].astype(np.float32)
        out[f'{name}/rms'] = np.sqrt((y.astype(np.float64) ** 2).mean(axis=1))
        out[f'{name}/meta'] = np.array([B, T, int(nsf), stride, hop], np.int64)
        print(name, y.shape, 'rms', out[f'{name}/rms'].mean())
    np.savez_compressed(os.path.join(OUT, 'generator_extra.npz'), **out)


GRAD_STRIDE, DISC_GRAD_STRIDE = 7, 633     # gradients are stored subsampled plus their exact L2 norm (keeps each fixture under 1 MB)


def grad_stride(numel, stride):
    return 1 if numel <= 4096 else stride


def _pack_grads(out, prefix, named_grads, stride=GRAD_STRIDE):
    for k, g in named_grads:
        g = g.detach().double().reshape(-1)
        out[f'{prefix}/{k}/norm'] = np.float64(g.norm())
        out[f'{prefix}/{k}/sub'] = g[::grad_stride(g.numel(), stride)].float().numpy()


def gen_generator_grads():
    """Parameter gradients by torch autograd through the REFERENCE generator modules (weight norm live, not folded):
    d sum(y * cot) / d every parameter, small configs (ResBlock1 NSF, ResBlock2 NSF)."""
    R.install()
    out = {}
    for name, cfg, B, T in (('small_nsf', None, 2, 24), ('small_rb2', 'small_rb2', 2, 24)):
        h = S.small_config(True) if cfg is None else extra_config(cfg, True)
        hop = int(np.prod(h['upsample_rates']))
        sd = S.make_generator_state_dict(h, SEED)
        mel, f0 = S.make_mel_f0(B, T, SEED)
        ri, nz = S.make_nsf_noise(B, T * hop, SEED)
        cot = torch.randn(B, 1, T * hop, generator=torch.Generator().manual_seed(7))
        model = R.build_generator(h, sd, fold=False).train()
        with R.injected_noise(ri, nz):
            y = model(mel, f0)
        (y * cot).sum().backward()
        _pack_grads(out, name, [(k, p.grad) for k, p in model.named_parameters()])
        out[f'{name}/y_sub'] = y.detach().numpy()[:, 0, ::3].astype(np.float32)
        print(name, 'params', len(list(model.parameters())))
    np.savez_compressed(os.path.join(OUT, 'generator_grads.npz'), **out)


def gen_losses_extra():
    """use_mel_loss STFT loss (modules/parallel_wavegan/stft_loss.py:13-100), the vocoder_denoise_c post-filter
    (vocoders/vocoder_utils.py:7-15) and save_wav's float -> int16 conversion (utils/audio.py:11-16)."""
    import tempfile
    R.install()
    from utils.hparams import hparams as ref_hp
    from modules.parallel_wavegan.stft_loss import MultiResolutionSTFTLoss as MelMR
    from vocoders.vocoder_utils import denoise
    from utils.audio import save_wav
    from scipy.io import wavfile
    out = {}
    y = S.make_wave_batch(2, 8192, seed=SEED)
    x = (y + 0.05 * S.make_wave_batch(2, 8192, seed=SEED + 1)).clamp(-1, 1)
    with R.legacy_stft(), R.cpu_cuda(), torch.no_grad():
        m = MelMR(use_mel_loss=True)
        sc, mag = m(x, y)
        out['mr_stft_mel/sc_mag'] = np.array([float(sc), float(mag)], np.float64)
        per = []
        for f in m.stft_losses:
            s1, m1 = f(x, y)
            per += [float(s1), float(m1)]
        out['mr_stft_mel/per_resolution'] = np.array(per, np.float64)
    xg = x.clone().requires_grad_(True)
    with R.legacy_stft(), R.cpu_cuda():
        sc, mag = MelMR(use_mel_loss=True)(xg, y)
        (sc + mag).backward()
    out['mr_stft_mel/dx_norm'] = np.float64(xg.grad.double().norm())
    out['mr_stft_mel/dx_sub'] = xg.grad.numpy()[:, ::5].astype(np.float32)
    for win in (512, 1024):
        ref_hp.update({'fft_size': 1024, 'hop_size': 256, 'win_size': win})
        wav = S.make_clip(256 * 40, seed=SEED + 3)
        out[f'denoise/win{win}'] = np.asarray(denoise(wav, v=0.1), np.float32)
    wav = S.make_clip(4000, seed=SEED + 4) * 1.7
    wav = np.clip(wav, -1.0, 1.0).astype(np.float32)
    for norm in (False, True):
        with tempfile.TemporaryDirectory() as d:
            fn = os.path.join(d, 'a.wav')
            save_wav(wav.copy(), fn, 22050, norm=norm)
            sr, data = wavfile.read(fn)
        assert sr == 22050 and data.dtype == np.int16
        out[f'save_wav/int16_norm{int(norm)}'] = data
    np.savez_compressed(os.path.join(OUT, 'losses_extra.npz'), **out)
    print('losses_extra.npz', out['mr_stft_mel/sc_mag'], out['denoise/win512'].shape)


def gen_discriminators_train():
    """Training-mode discriminators from the reference modules: (i) MSD in train() mode -- torch's spectral_norm runs
    one power iteration per forward of every DiscriminatorS[0] conv (hifigan.py:261,294), so two MSD forwards =
    four iterations: logits and the u buffers after each forward; (ii) parameter gradients of the D loss and
    d(G adversarial + feature loss)/d y_hat by autograd through the reference MPD / MSD."""
    R.install()
    from utils.hparams import hparams as ref_hp
    ref_hp['hop_size'] = 256
    from modules.hifigan.hifigan import (MultiPeriodDiscriminator, MultiScaleDiscriminator, discriminator_loss, feature_loss,
                                         generator_loss)
    out = {}
    y = S.make_wave_batch(2, 8192, seed=SEED)[:, None]
    y_hat = (y + 0.1 * S.make_wave_batch(2, 8192, seed=SEED + 5)[:, None]).clamp(-1, 1)
    for name, cls, sd in (('mpd', MultiPeriodDiscriminator, S.make_mpd_state_dict(SEED)),
                          ('msd', MultiScaleDiscriminator, S.make_msd_state_dict(SEED))):
        m = cls()
        m.load_state_dict(sd, strict=True)
        m.train()
        # ---- forward 1 (+ D-loss gradients), then forward 2 on the updated u / v
        rs, gs, fr, fg = m(y, y_hat)
        r_loss, g_loss = discriminator_loss(rs, gs)
        (r_loss + g_loss).backward()
        out[f'{name}/d_loss'] = np.array([float(r_loss), float(g_loss)], np.float64)
        _pack_grads(out, f'{name}/d_grad', [(k, p.grad) for k, p in m.named_parameters()], DISC_GRAD_STRIDE)
        for i, (r, g) in enumerate(zip(rs, gs)):
            out[f'{name}/fwd1/logit_r{i}'], out[f'{name}/fwd1/logit_g{i}'] = r.detach().numpy(), g.detach().numpy()
        if name == 'msd':
            for k, b in m.named_buffers():
                if k.endswith('weight_u'):
                    out[f'{name}/fwd1/{k}'] = b.detach().numpy().copy()
        m.zero_grad()
        with torch.no_grad():
            rs2, gs2, _, _ = m(y, y_hat)
        for i, (r, g) in enumerate(zip(rs2, gs2)):
            out[f'{name}/fwd2/logit_r{i}'], out[f'{name}/fwd2/logit_g{i}'] = r.numpy(), g.numpy()
        if name == 'msd':
            for k, b in m.named_buffers():
                if k.endswith('weight_u'):
                    out[f'{name}/fwd2/{k}'] = b.detach().numpy().copy()
        # ---- generator side: d (generator_loss + feature_loss) / d y_hat with the discriminator frozen (eval-mode
        # spectral norm so the fixture does not depend on how many iterations ran before)
        m2 = cls()
        m2.load_state_dict(sd, strict=True)
        m2.eval()
        for p in m2.parameters():
            p.requires_grad_(False)
        yh = y_hat.clone().requires_grad_(True)
        rs, gs, fr, fg = m2(y, yh)
        lg = generator_loss(gs) + feature_loss(fr, fg)
        lg.backward()
        out[f'{name}/g_loss'] = np.float64(lg)
        out[f'{name}/g_dyhat_norm'] = np.float64(yh.grad.double().norm())
        out[f'{name}/g_dyhat_sub'] = yh.grad.numpy()[:, 0, ::5].astype(np.float32)
        print(name, out[f'{name}/d_loss'], float(lg))
    np.savez_compressed(os.path.join(OUT, 'discriminators_train.npz'), **out)


WN_CASES = {
    # name: (hidden, kernel, dilation_rate, n_layers, gin, B, T)      GlobalFVAE decoder / encoder shapes (vae_models.py:81-146)
    'fvae_dec': (192, 5, 1, 4, 0, 2, 100),
    'fvae_enc_cond': (192, 5, 1, 8, 256, 2, 61),
    'dilated_cond': (64, 3, 2, 3, 32, 1, 300),
}


def gen_wn():
    """WN outputs of the reference class itself (modules/fastspeech/fs2_vae.py:19-94), weight-normed then folded."""
    R.install()
    import contextlib
    import io
    from modules.fastspeech.fs2_vae import WN
    out = {}
    for name, (H, K, dr, L, gin, B, T) in WN_CASES.items():
        sd = S.make_wn_state_dict(H, K, L, gin, SEED)
        x, mask, g = S.make_wn_inputs(B, T, H, gin, SEED)
        m = WN(H, K, dr, L, gin_channels=gin)
        m.load_state_dict(sd, strict=True)
        with contextlib.redirect_stdout(io.StringIO()):
            m.remove_weight_norm()
        m.eval()
        with torch.no_grad():
            y = m(x, mask, g)
        out[f'{name}/y'] = y.numpy().astype(np.float32)
        out[f'{name}/params'] = np.array([H, K, dr, L, gin, B, T], np.int64)
    np.savez_compressed(os.path.join(OUT, 'wn.npz'), **out)
    print('wn.npz', {k: v.shape for k, v in out.items() if k.endswith('/y')})


FVAE_DEC_CASES = {
    # name: (latent, hidden, out, kernel, n_layers, gin, B, T, global latent)   vae_global_mle_eng: hidden 192, latent 128, k 5, dec 4 layers
    'global_dec': (128, 192, 80, 5, 4, 256, 2, 120, True),
    'local_dec_nocond_mask1': (16, 64, 80, 3, 2, 0, 1, 52, False),
}


def gen_fvae_decoder():
    """Mel decoder outputs of the reference classes (FVAEDecoder fs2_vae.py:130-152, GlobalFVAEDecoder vae_models.py:108-128)."""
    R.install()
    import contextlib
    import io
    from modules.fastspeech.fs2_vae import FVAEDecoder
    from modules.voice_conversion.vae_models import GlobalFVAEDecoder
    out = {}
    for name, (lat, H, oc, K, L, gin, B, T, glob) in FVAE_DEC_CASES.items():
        sd = S.make_fvae_decoder_state_dict(lat, H, oc, K, L, gin, 4, SEED)
        _, mask, g = S.make_wn_inputs(B, T, H, gin, SEED)
        rs = np.random.RandomState(SEED + 5)
        z = torch.from_numpy(rs.randn(B, lat, 1 if glob else T // 4).astype(np.float32))
        m = (GlobalFVAEDecoder if glob else FVAEDecoder)(lat, H, oc, K, L, gin, strides=[4])
        m.load_state_dict(sd, strict=True)
        with contextlib.redirect_stdout(io.StringIO()):
            m.wn.remove_weight_norm()
        m.eval()
        with torch.no_grad():
            y = m(z, mask if glob else 1, g)             # the reference passes x_mask = 1 at inference (fs2_vae.py:213)
        out[f'{name}/y'] = y.numpy().astype(np.float32)
        out[f'{name}/params'] = np.array([lat, H, oc, K, L, gin, B, T, int(glob)], np.int64)
    np.savez_compressed(os.path.join(OUT, 'fvae_decoder.npz'), **out)
    print('fvae_decoder.npz', {k: v.shape for k, v in out.items() if k.endswith('/y')})


def gen_fvae_encoder():
    """(m, logs) of the reference GlobalFVAEEncoder in eval mode (vae_models.py:81-106; hidden 192, latent 128, 8 WN layers)."""
    R.install()
    import contextlib
    import io
    from modules.voice_conversion.vae_models import GlobalFVAEEncoder
    cin, H, lat, K, L, gin, B, T = 80, 192, 128, 5, 8, 256, 2, 400
    sd = S.make_fvae_encoder_state_dict(cin, H, lat, K, L, gin, 4, SEED)
    rs = np.random.RandomState(SEED + 11)
    x = torch.from_numpy(rs.randn(B, cin, T).astype(np.float32))
    mask = torch.ones(B, 1, T)
    mask[1, :, T - 36:] = 0
    g = torch.from_numpy(rs.randn(B, gin, T // 4).astype(np.float32))
    m = GlobalFVAEEncoder(cin, H, lat, K, L, gin, strides=[4])
    m.load_state_dict(sd, strict=True)
    with contextlib.redirect_stdout(io.StringIO()):
        m.wn.remove_weight_norm()
    m.eval()
    with torch.no_grad():
        z, mq, logs, xm = m(x * mask, mask, g)
    out = {'m': mq.numpy(), 'logs': logs.numpy(), 'mask_len': xm.sum(-1).numpy(), 'params': np.array([cin, H, lat, K, L, gin, B, T], np.int64)}
    np.savez_compressed(os.path.join(OUT, 'fvae_encoder.npz'), **out)
    print('fvae_encoder.npz', {k: v.shape for k, v in out.items()})


def gen_global_fvae():
    """x_recon / loss_kl / m_q / logs_q of the reference GlobalFVAE (vae_models.py:130-146, TMPFVAE.forward :11-44) in eval mode with the
    posterior noise replaced by zeros (z_q = m_q), at the vae_global_mle_eng sizes."""
    R.install()
    import contextlib
    import io
    from modules.voice_conversion.vae_models import GlobalFVAE
    io_c, H, lat, K, Le, Ld, gin, B, T = 80, 192, 128, 5, 8, 4, 256, 2, 240
    sd = S.make_global_fvae_state_dict(io_c, H, lat, K, Le, Ld, gin, 4, SEED)
    rs = np.random.RandomState(SEED + 23)
    x = torch.from_numpy(rs.randn(B, io_c, T).astype(np.float32))
    mask = torch.ones(B, 1, T)
    mask[1, :, T - 40:] = 0
    g = torch.from_numpy(rs.randn(B, gin, T).astype(np.float32))
    m = GlobalFVAE(io_c, H, lat, K, Le, Ld, gin, [4], False)
    m.load_state_dict(sd, strict=True)
    with contextlib.redirect_stdout(io.StringIO()):
        m.encoder.wn.remove_weight_norm(), m.decoder.wn.remove_weight_norm()
    m.eval()
    orig = torch.randn_like
    torch.randn_like = lambda t, **k: torch.zeros_like(t)
    try:
        with torch.no_grad():
            x_recon, loss_kl, _, m_q, logs_q, xm, z_q = m(x * mask, mask, g, infer=False)
    finally:
        torch.randn_like = orig
    out = {'x_recon': x_recon.numpy(), 'loss_kl': np.float64(loss_kl), 'm_q': m_q.numpy(), 'logs_q': logs_q.numpy(),
           'params': np.array([io_c, H, lat, K, Le, Ld, gin, B, T], np.int64)}
    np.savez_compressed(os.path.join(OUT, 'global_fvae.npz'), **out)
    print('global_fvae.npz', {k: np.shape(v) for k, v in out.items()})


def gen_vc_asr():
    """h_content of the reference VCASR (vc_modules.py:56-80; hidden 256, mel_strides [2, 1, 1], 2 conformer layers, asr_last_norm false)
    in eval mode on a random-init model whose state_dict is stored seed-reproducibly by neuralsvb_b200/utils/synthetic.py."""
    R.install()
    from utils.hparams import hparams
    hparams.update({'hidden_size': 256, 'asr_enc_layers': 2, 'asr_dec_layers': 2, 'mel_strides': [2, 1, 1], 'asr_enc_type': 'conformer',
                    'asr_last_norm': False, 'dropout': 0.1, 'enc_ffn_kernel_size': 9, 'num_heads': 2, 'enc_layers': 4, 'dec_layers': 4,
                    'ffn_hidden_size': 1024, 'ffn_padding': 'SAME', 'ffn_act': 'gelu', 'dec_ffn_kernel_size': 9, 'use_pos_embed': True})
    from modules.voice_conversion.vc_modules import VCASR
    m = VCASR(80, 80)
    sd = S.make_vc_asr_state_dict(SEED)
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all(k.startswith(('asr_decoder', 'token_embed')) for k in missing.missing_keys), missing
    m.eval()
    mel = S.make_vc_asr_mel(2, 157, SEED)
    with torch.no_grad():
        h = m(mel)['h_content']
    out = {'h_content': h.numpy(), 'params': np.array([2, 157], np.int64)}
    np.savez_compressed(os.path.join(OUT, 'vc_asr.npz'), **out)
    print('vc_asr.npz', h.shape, float(h.abs().max()))


SVB_HPARAMS = {'hidden_size': 256, 'audio_num_mel_bins': 80, 'asr_enc_layers': 2, 'asr_dec_layers': 2, 'mel_strides': [2, 1, 1],
               'asr_enc_type': 'conformer', 'asr_last_norm': False, 'dropout': 0.1, 'enc_ffn_kernel_size': 9, 'num_heads': 2,
               'enc_layers': 4, 'dec_layers': 4, 'ffn_hidden_size': 1024, 'ffn_padding': 'SAME', 'ffn_act': 'gelu', 'dec_ffn_kernel_size': 9,
               'use_pos_embed': True, 'latent_size': 128, 'fvae_enc_dec_hidden': 192, 'fvae_kernel_size': 5, 'fvae_enc_n_layers': 8,
               'fvae_dec_n_layers': 4, 'frames_multiple': 4, 'use_prior_glow': False}


def gen_svb_vae():
    """a2a / p2p / a2p outputs of the reference MleSVBVAE (svb_vae.py:251-312) in eval mode at the vae_global_mle_eng sizes, posterior
    noise replaced by zeros; also the name / shape listing of its state_dict (the drop-in class must expose the same keys)."""
    R.install()
    from utils.hparams import hparams
    hparams.update(SVB_HPARAMS)
    from modules.voice_conversion.svb_vae import MleSVBVAE
    m = MleSVBVAE(80)
    sd = S.make_svb_state_dict(SEED)
    res = m.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys and all(k.startswith(('vc_asr.asr_decoder', 'vc_asr.token_embed')) for k in res.missing_keys), res
    for wn in (m.vae_model.encoder.wn, m.vae_model.decoder.wn):
        wn.remove_weight_norm()
    m.eval()
    batch = S.make_svb_batch(2, 96, 120, SEED)
    orig = torch.randn_like
    torch.randn_like = lambda t, **k: torch.zeros_like(t)
    try:
        with torch.no_grad():
            ret = m(**batch, infer=False, concurrent_ways=['a2a', 'p2p', 'a2p'])
    finally:
        torch.randn_like = orig
    keys = [k for k in MleSVBVAE(80).state_dict().keys() if not k.startswith(('vc_asr.asr_decoder', 'vc_asr.token_embed'))]
    shapes = MleSVBVAE(80).state_dict()
    out = {'a2p_mel': ret['a2p']['mel_out'].numpy(), 'a2p_mle': np.float64(ret['a2p']['mle']), 'a2a_mel': ret['a2a']['mel_out'].numpy(),
           'p2p_m_q': ret['p2p']['m_q'].numpy(), 'a2a_kl': np.float64(ret['a2a']['kl']),
           'state_keys': np.array(keys), 'state_shapes': np.array([','.join(str(d) for d in shapes[k].shape) for k in keys])}
    np.savez_compressed(os.path.join(OUT, 'svb_vae.npz'), **out)
    print('svb_vae.npz', out['a2p_mel'].shape, float(np.abs(out['a2p_mel']).max()), len(keys), 'state keys')


HPARAMS_CASES = [('egs/egs_bases/tts/vocoder/hifigan.yaml', 'hop_size=128'),
                 ('egs/datasets/audio/PopBuTFy/vae_global_mle_eng.yaml', 'hop_size=128')]


def gen_hparams():
    """The reference's set_hparams (utils/hparams.py) on base_config chains of its egs/ tree: every YAML file it opened, stored
    parsed (the resolver reads them with yaml.safe_load), and the dict it returned for each (config, --hparams) case."""
    import builtins
    import importlib.util
    import json
    import yaml
    spec = importlib.util.spec_from_file_location('ref_hparams', os.path.join(R.REF_ROOT, 'utils', 'hparams.py'))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    opened = []
    ref.open = lambda fn, *a, **k: (opened.append(fn), builtins.open(fn, *a, **k))[1]
    cwd = os.getcwd()
    os.chdir(R.REF_ROOT)
    try:
        cases = [{'config': cfg, 'hparams_str': hs,
                  'resolved': ref.set_hparams(cfg, hparams_str=hs, print_hparams=False, global_hparams=False)}
                 for cfg, hs in HPARAMS_CASES]
        files = {fn: yaml.safe_load(open(fn)) for fn in sorted(set(opened))}
    finally:
        os.chdir(cwd)
    out = {'files': files, 'cases': cases}
    assert json.loads(json.dumps(out)) == out, 'a resolved value does not survive JSON'
    with open(os.path.join(OUT, 'hparams.json'), 'w') as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write('\n')
    print('hparams.json', len(files), 'YAML files,', [len(c['resolved']) for c in cases], 'resolved keys')


def main():
    if not R.available():
        sys.exit('gen_golden needs /root/reference (build container only)')
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    warnings.simplefilter('ignore')
    which = sys.argv[1:] or ['frontend', 'generator', 'losses', 'discriminators', 'discriminators_cond', 'generator_extra',
                             'generator_grads', 'losses_extra', 'discriminators_train', 'wn', 'fvae_decoder', 'fvae_encoder', 'global_fvae', 'vc_asr', 'svb_vae', 'hparams']
    for w in which:
        globals()[f'gen_{w}']()


if __name__ == '__main__':
    main()
