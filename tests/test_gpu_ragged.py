"""-m gpu: ragged batches through the generator (svb_gen_forward_ragged / HifiGanGenerator.forward(lengths=...) /
HifiGAN.spec2wav_ragged).  A clip's samples must be bit-identical to a forward of that clip alone: row arithmetic does
not depend on where a tile sits or which clips share a launch (test_batch_independence_and_causal_extent)."""
import contextlib
import ctypes
import io

import numpy as np
import pytest
import torch

from neuralsvb_b200 import _native
from neuralsvb_b200.modules.hifigan.hifigan import HifiGanGenerator
from neuralsvb_b200.utils import synthetic as S
from oracle import hifigan as O
from tests import gpu_util as U

pytestmark = pytest.mark.gpu

LENS = [1, 7, 37, 128, 129, 255, 256, 300]          # tile edges, a 1-frame clip, clips shorter than conv_pre's halo
CASES = [(cfg, p) for cfg in ('hop256', 'small') for p in ('fp32', 'bf16x3')]


def _fresh(h, precision):
    m = HifiGanGenerator(h, precision=precision)
    m.load_state_dict(S.make_generator_state_dict(h, U.SEED), strict=True)
    with contextlib.redirect_stdout(io.StringIO()):
        m.remove_weight_norm()
    return m.eval().to('cuda:0')


def _inputs(h, lens, nsf=True, fill=None):
    hop = int(np.prod(h['upsample_rates']))
    B, T = len(lens), max(lens)
    mel, f0 = S.make_mel_f0(B, T, U.SEED)
    ri, nz = S.make_nsf_noise(B, T * hop, U.SEED)
    if fill is not None:                             # poison everything past each clip's length
        for b, L in enumerate(lens):
            mel[b, :, L:] = fill
            f0[b, L:] = fill
            nz[b, L * hop:] = fill
    return hop, mel.cuda(), (f0.cuda() if nsf else None), ri.cuda(), nz.cuda()


def _single(m, mel, f0, ri, nz, b, L, hop):
    return m(mel[b:b + 1, :, :L].contiguous(), None if f0 is None else f0[b:b + 1, :L].contiguous(),
             rand_ini=ri[b:b + 1].contiguous(), noise=nz[b:b + 1, :L * hop].contiguous())


def _check_clips(y, m, mel, f0, ri, nz, lens, hop):
    for b, L in enumerate(lens):
        ref = _single(m, mel, f0, ri, nz, b, L, hop)
        assert torch.equal(y[b:b + 1, :, :L * hop], ref), (b, L)
        assert not y[b, :, L * hop:].any(), (b, L)


@pytest.mark.parametrize('cfg,precision', CASES)
def test_ragged_equals_each_clip_alone(cfg, precision):
    h = U.config(cfg, True)
    m = U.cuda_generator(cfg, True, precision)
    hop, mel, f0, ri, nz = _inputs(h, LENS)
    with torch.no_grad():
        y = m(mel, f0, rand_ini=ri, noise=nz, lengths=LENS)
        assert tuple(y.shape) == (len(LENS), 1, max(LENS) * hop)
        _check_clips(y, m, mel, f0, ri, nz, LENS, hop)


@pytest.mark.parametrize('cfg,precision', CASES)
def test_padding_is_never_read(cfg, precision):
    h = U.config(cfg, True)
    m = U.cuda_generator(cfg, True, precision)
    lens = [5, 130, 64]
    with torch.no_grad():
        hop, *clean = _inputs(h, lens)
        y0 = m(*clean[:2], rand_ini=clean[2], noise=clean[3], lengths=lens)
        for fill in (float('nan'), 1e4, -1e4):
            _, mel, f0, ri, nz = _inputs(h, lens, fill=fill)
            y = m(mel, f0, rand_ini=ri, noise=nz, lengths=torch.tensor(lens, device='cuda'))
            assert torch.isfinite(y).all() and torch.equal(y, y0), fill


@pytest.mark.parametrize('cfg,precision', CASES)
def test_stale_tails_of_a_longer_call_are_cleared(cfg, precision):
    h = U.config(cfg, True)
    lens_short = [3, 129, 40, 1]
    B, T = len(lens_short), 260
    hop = int(np.prod(h['upsample_rates']))
    mel, f0 = S.make_mel_f0(B, T, U.SEED)
    ri, nz = S.make_nsf_noise(B, T * hop, U.SEED)
    mel, f0, ri, nz = mel.cuda(), f0.cuda(), ri.cuda(), nz.cuda()
    with torch.no_grad():
        ref = _fresh(h, precision)(mel, f0, rand_ini=ri, noise=nz, lengths=lens_short)
        m = _fresh(h, precision)
        m(mel, f0, rand_ini=ri, noise=nz, lengths=[T, T - 1, T, T - 5])          # every clip long
        assert torch.equal(m(mel, f0, rand_ini=ri, noise=nz, lengths=lens_short), ref)
        m(mel, f0, rand_ini=ri, noise=nz)                                           # an equal-length forward at T
        assert torch.equal(m(mel, f0, rand_ini=ri, noise=nz, lengths=lens_short), ref)


@pytest.mark.parametrize('precision', ['fp32', 'bf16x3'])
def test_ragged_against_the_oracle(precision):
    h = U.config('hop256', True)
    lens = [9, 40, 23]
    m = U.cuda_generator('hop256', True, precision)
    hop, mel, f0, ri, nz = _inputs(h, lens)
    w = O.fold_weight_norm(S.make_generator_state_dict(h, U.SEED))
    with torch.no_grad():
        y = m(mel, f0, rand_ini=ri, noise=nz, lengths=lens).cpu().numpy()[:, 0]
        for b, L in enumerate(lens):
            y_o = O.generator_forward(w, h, mel[b:b + 1, :, :L].cpu(), f0[b:b + 1, :L].cpu(), ri[b:b + 1].cpu(),
                                      nz[b:b + 1, :L * hop].cpu()).numpy()[0, 0]
            assert U.rms(y[b, :L * hop], y_o) < 1e-4, (b, U.rms(y[b, :L * hop], y_o))


@pytest.mark.parametrize('cfg,precision', CASES)
def test_uniform_lengths_equal_the_plain_forward(cfg, precision):
    h = U.config(cfg, True)
    m = U.cuda_generator(cfg, True, precision)
    lens = [70] * 4
    hop, mel, f0, ri, nz = _inputs(h, lens)
    with torch.no_grad():
        assert torch.equal(m(mel, f0, rand_ini=ri, noise=nz, lengths=lens), m(mel, f0, rand_ini=ri, noise=nz))
        assert torch.equal(m(mel, f0, seed=5, lengths=lens), m(mel, f0, seed=5))
        # Philox noise is keyed by (sample, clip): a clip does not change when its neighbour's length does
        a = m(mel, f0, seed=5, lengths=[70, 20, 70, 33])
        b = m(mel, f0, seed=5, lengths=[70, 61, 70, 2])
        full = m(mel, f0, seed=5)
        for i in (0, 2):
            assert torch.equal(a[i], b[i]) and torch.equal(a[i], full[i])
        assert torch.equal(a[1, :, :20 * hop], m(mel, f0, seed=5, lengths=[70, 20, 1, 1])[1, :, :20 * hop])


@pytest.mark.parametrize('precision', ['fp32', 'bf16x3'])
def test_non_nsf_resblock2_and_unmerged_schedule(precision, monkeypatch):
    lens = [33, 1, 140]
    h = U.config('hop256', False)
    m = U.cuda_generator('hop256', False, precision)
    hop, mel, _, ri, nz = _inputs(h, lens, nsf=False)
    with torch.no_grad():
        y = m(mel, lengths=lens)
        for b, L in enumerate(lens):
            assert torch.equal(y[b:b + 1, :, :L * hop], m(mel[b:b + 1, :, :L].contiguous()))
            assert not y[b, :, L * hop:].any()
        h2 = S.hifigan_config()
        h2['resblock'] = '2'
        h2['resblock_dilation_sizes'] = [[1, 3], [1, 3], [1, 3]]
        m2 = _fresh(h2, precision)
        hop, mel, f0, ri, nz = _inputs(h2, lens)
        _check_clips(m2(mel, f0, rand_ini=ri, noise=nz, lengths=lens), m2, mel, f0, ri, nz, lens, hop)
        monkeypatch.setenv('SVB_MERGE', '0')             # read by svb_gen_create: a handle with one launch per conv
        h3 = S.hifigan_config()
        m3 = _fresh(h3, precision)
        hop, mel, f0, ri, nz = _inputs(h3, lens)
        y3 = m3(mel, f0, rand_ini=ri, noise=nz, lengths=lens)
        _check_clips(y3, m3, mel, f0, ri, nz, lens, hop)
        assert torch.equal(y3, U.cuda_generator('hop256', True, precision)(mel, f0, rand_ini=ri, noise=nz, lengths=lens))


def test_host_path_matches_batch_and_device_paths():
    from neuralsvb_b200.utils.hparams import hparams
    from neuralsvb_b200.vocoders.hifigan import HifiGAN
    h = U.config('hop256', True)
    m = U.cuda_generator('hop256', True, 'bf16x3')
    voc = HifiGAN.from_model(m, h)
    hop = 256
    hparams['vocoder_denoise_c'] = 0.0
    mel, f0 = S.make_mel_f0(3, 50, U.SEED)
    mels = [mel[b].T.numpy() for b in range(3)]
    f0s = [f0[b].numpy() for b in range(3)]
    got = voc.spec2wav_ragged(mels, f0s, seed=9)                      # equal lengths: the batch call, clip by clip
    want = voc.spec2wav_batch(np.stack(mels), np.stack(f0s), seed=9)
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    lens = [50, 13, 1]
    mels_r = [mels[b][:L] for b, L in enumerate(lens)]
    f0s_r = [f0s[b][:L] for b, L in enumerate(lens)]
    got = voc.spec2wav_ragged(mels_r, f0s_r, seed=9)
    with torch.no_grad():
        dev = m(mel.cuda(), f0.cuda(), seed=9, lengths=lens).cpu().numpy()[:, 0]
    for b, L in enumerate(lens):
        assert got[b].dtype == np.float32 and got[b].shape == (L * hop,)
        assert np.array_equal(got[b], dev[b, :L * hop])
    nomel = voc.spec2wav_ragged(mels_r, seed=9)                       # the non-NSF call on an NSF model
    assert [len(w) for w in nomel] == [L * hop for L in lens] and all(np.isfinite(w).all() for w in nomel)
    from oracle import frontend as FE
    for norm in (False, True):                                        # norm: each clip's peak over its own samples
        q = voc.spec2wav_ragged(mels_r, f0s_r, seed=9, int16=True, norm=norm)
        for b in range(3):
            assert q[b].dtype == np.int16 and np.array_equal(q[b], FE.float_to_int16(got[b], norm)), (b, norm)
    hparams['vocoder_denoise_c'] = 0.1
    try:
        with pytest.raises(ValueError, match='exclusive'):
            voc.spec2wav_ragged(mels_r, f0s_r, int16=True)
    finally:
        hparams['vocoder_denoise_c'] = 0.0


def test_training_rejects_ragged_and_flops_count_valid_rows():
    h = U.config('small', True)
    m = U.cuda_generator('small', True, 'bf16x3')
    lib = _native.lib()
    lens = [40, 10, 25, 5]
    hop, mel, f0, ri, nz = _inputs(h, lens)
    with torch.no_grad():
        m(mel, f0, rand_ini=ri, noise=nz)
        g = m.native_handle(mel.device)
        full = lib.svb_gen_last_flops(g)
        m(mel, f0, rand_ini=ri, noise=nz, lengths=lens)
        ragged = lib.svb_gen_last_flops(g)
    assert ragged == pytest.approx(full * sum(lens) / (len(lens) * max(lens)), rel=1e-9)
    # the C ABI: a handle in training mode refuses a ragged batch
    tm = _fresh(h, 'bf16x3')
    tg = tm.native_handle(mel.device)
    y = torch.empty(len(lens), 1, max(lens) * hop, device='cuda')
    ln = np.array(lens, np.int32)
    _native.check(lib.svb_gen_set_training(tg, 1), 'set_training')
    rc = lib.svb_gen_forward_ragged(tg, _native.ptr(mel), _native.ptr(f0), ln.ctypes.data_as(ctypes.c_void_p), None, None,
                                    ctypes.c_uint64(1), len(lens), max(lens), _native.ptr(y), None)
    assert rc == -1 and b'inference only' in lib.svb_last_error()
    tm.train()
    with pytest.raises(NotImplementedError):
        tm(mel, f0, lengths=lens)
