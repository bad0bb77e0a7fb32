"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, and
exports every symbol include/svb_vocoder.h declares.  No compute calls (no GPU here)."""
import ctypes
import os

import pytest

from neuralsvb_b200 import _native


@pytest.fixture(scope='module')
def built():
    try:
        return _native.build()
    except RuntimeError as e:          # no nvcc on this box: the prebuilt library must already be there
        if os.path.exists(_native.LIB_PATH):
            return _native.LIB_PATH
        pytest.fail(str(e))


def test_library_exports_every_declared_symbol(built):
    l = ctypes.CDLL(built)
    declared = _native.declared_symbols()
    assert len(declared) >= 15
    missing = [s for s in declared if not hasattr(l, s)]
    assert not missing, f'declared in include/svb_vocoder.h but not exported: {missing}'


def test_binding_covers_every_declared_symbol():
    declared = set(_native.declared_symbols())
    bound = set(_native._PROTOS)
    assert declared <= bound, f'no ctypes prototype for {sorted(declared - bound)}'


def test_abi_version_and_error_string(built):
    l = _native.lib()
    assert l.svb_abi_version() == 1
    assert isinstance(l.svb_last_error(), bytes)


def test_struct_layout_matches_header():
    # 3 + 8 + 8 + 2 + 4 + 1 + 16 + 3 int32 fields
    assert ctypes.sizeof(_native.GenConfig) == 4 * (3 + 8 + 8 + 2 + 4 + 1 + 16 + 3)
    assert ctypes.sizeof(_native.StftConfig) == 4 * 9


def test_argument_validation_without_gpu(built):
    l = _native.lib()
    # null config -> SVB_ERR_INVALID before any CUDA call
    assert l.svb_stft_num_frames(None, 100) < 0
    c = _native.StftConfig(1024, 256, 512, _native.PAD_CENTER_ZERO, _native.OUT_LOG10_MEL, 0, 80, 1, 1e-10)
    assert l.svb_stft_num_frames(ctypes.byref(c), 44100) == 173          # 1 + n // hop
    assert l.svb_stft_num_frames(ctypes.byref(c), 1000) == 4
    c.pad_mode = _native.PAD_HALF_REFLECT
    assert l.svb_stft_num_frames(ctypes.byref(c), 32768) == 128          # T_wav / hop exactly
    c.n_fft = 1000                                                      # not a power of two
    rc = l.svb_stft_forward(ctypes.byref(c), None, 1, 100, None, None, None)
    assert rc == -1 and b'power of two' in l.svb_last_error()


def test_product_fails_loudly_without_cuda(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: False)        # behave as without a CUDA device, whether or not one is present
    from neuralsvb_b200.modules.hifigan.hifigan import HifiGanGenerator
    from neuralsvb_b200.utils import synthetic as S
    h = S.small_config()
    m = HifiGanGenerator(h)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m(torch.zeros(1, 80, 8))
    from neuralsvb_b200.vocoders.hifigan import HifiGAN
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        HifiGAN.wav2spec(S.make_clip(2048), hp=S.hifigan_config())


def test_training_entry_points_validate_arguments_without_gpu(built):
    """The backward / training half of the ABI rejects bad arguments before any CUDA call (negative svb_status, message set)."""
    l = _native.lib()
    f = ctypes.c_float
    assert l.svb_gen_set_training(None, 1) < 0 and b'not finalized' in l.svb_last_error()
    assert l.svb_gen_backward(None, None, None) < 0
    assert l.svb_gen_grad_numel(None, b'conv_pre.weight') == -1
    assert l.svb_weight_norm_backward(None, None, None, 4, 4, None, None, None) < 0
    assert l.svb_conv_nct_backward(None, None, None, None, 1, 1, 1, 8, 1, 3, 1, 1, 1, 1, f(0.1), None, None, None, None, None) < 0
    assert l.svb_loss_grad_dev(None, None, 0, f(1.0), None, None, 8, 0, None) < 0
    assert l.svb_cond_net_forward(None, None, None, 1, 80, 8, 512, 256, 128, None, None) < 0
    h = ctypes.c_void_p()
    # 33 -> 64 channels is not a tensor-core shape; a stride-1 layer needs 'same' padding
    assert l.svb_tc_layer_create(33, 64, 5, 1, 2, 3, 0, ctypes.byref(h)) < 0 and b'tensor-core shape' in l.svb_last_error()
    assert l.svb_tc_layer_create(64, 64, 5, 1, 1, 3, 0, ctypes.byref(h)) < 0 and b"'same' padding" in l.svb_last_error()
    assert l.svb_tc_layer_create(64, 64, 5, 3, 2, 0, 0, ctypes.byref(h)) < 0          # fp32 is not a tensor-core mode
    assert l.svb_tc_layer_out_len(None, 100) == -1
    c = _native.StftConfig(1024, 256, 512, _native.PAD_CENTER_ZERO, _native.OUT_MAG_RAW, 0, 0, 1, 0.0)
    assert l.svb_denoise(ctypes.byref(c), None, 1, 4096, f(0.1), None, None) < 0
    c.n_fft = 1000
    assert l.svb_stft_backward(ctypes.byref(c), None, 1, 4096, None, None, None, None) < 0 and b'power of two' in l.svb_last_error()


def _schedule(KS, has_res, accum, B, Tq, MT, col_blocks, chain_ordered, grid=148, Cin=128):
    import ctypes

    import numpy as np
    from neuralsvb_b200 import _native
    n = len(KS)
    arr = lambda v: np.ascontiguousarray(v, dtype=np.int32)
    ks, hr, ac = arr(KS), arr(has_res), arr(accum)
    cap = 200000
    items, off, bal = np.zeros((cap, 5), np.int32), np.zeros(grid + 1, np.int32), ctypes.c_double()
    cnt = _native.check(_native.lib().svb_tc_schedule_probe(n, ks.ctypes.data, hr.ctypes.data, ac.ctypes.data, Cin, B, Tq, MT, col_blocks,
                                                            int(chain_ordered), grid, items.ctypes.data, cap, off.ctypes.data, ctypes.byref(bal)),
                        'tc_schedule_probe')
    return items[:cnt], off, bal.value


def test_merged_launch_schedule_covers_every_tile_once():
    """Host logic of the merged ResBlock-chain launches (csrc/conv_tc.cu:tc_schedule), no GPU needed: the three chains of stage 1 of
    config 2 (C = 128: k 3 / 7 / 11, 16 clips x 8192 rows)."""
    import numpy as np
    items, off, bal = _schedule([3, 7, 11], [0, 0, 0], [0, 0, 0], 16, 8192, 2, 1, False)
    assert len(items) == 3 * 16 * 32 and off[0] == 0 and off[-1] == len(items)
    seen = set(map(tuple, items[:, :4]))
    assert len(seen) == len(items)                                           # no (layer, block, clip, row) twice
    for l in range(3):
        rows = items[items[:, 0] == l]
        assert sorted(map(tuple, rows[:, 2:4])) == [(b, t) for b in range(16) for t in range(0, 8192, 256)]
    assert (items[:, 4] == 2).all() and bal > 0.95
    assert (np.diff(off) <= 120).all()
    # a CTA alternates its layers instead of running them one after the other
    first = items[off[0]:off[1], 0]
    assert len(set(first[:3].tolist())) > 1


def test_chain_ordered_schedule_keeps_the_layers_of_a_tile_together():
    """The step that accumulates the three ResBlocks into the stage output: every CTA runs layers 0, 1, 2 of a tile back to back."""
    items, off, bal = _schedule([3, 7, 11], [1, 1, 1], [0, 1, 1], 16, 1024, 2, 2, True, Cin=256)
    assert len(items) == 3 * 16 * 4 * 2
    for c in range(len(off) - 1):
        mine = items[off[c]:off[c + 1]]
        assert len(mine) % 3 == 0
        for i in range(0, len(mine), 3):
            assert mine[i:i + 3, 0].tolist() == [0, 1, 2]
            assert (mine[i:i + 3, 1:] == mine[i, 1:]).all()                    # same column block, clip, row, tiles
    assert 0.8 < bal <= 1.0


def test_schedule_handles_an_odd_tile_count():
    items, off, bal = _schedule([3, 11], [0, 0], [0, 0], 3, 5 * 128 - 7, 2, 1, False, grid=8)
    tiles = items[:, 4]
    assert set(tiles.tolist()) == {1, 2}                                      # the last item of a clip has one tile
    assert int(tiles.sum()) == 2 * 3 * 5
