"""CPU-side checks of ragged batches (no GPU): the per-clip schedule of the merged tensor-core launches and the argument
checks of the ragged entry points, which run before any CUDA call."""
import ctypes

import numpy as np
import pytest

from neuralsvb_b200 import _native


@pytest.fixture(scope='module')
def lib():
    try:
        _native.build()
    except RuntimeError:
        pass
    return _native.lib()


def _schedule(lib, KS, has_res, accum, rows, MT, col_blocks, chain_ordered, grid=148, Cin=128):
    n = len(KS)
    arr = lambda v: np.ascontiguousarray(v, dtype=np.int32)
    ks, hr, ac, rw = arr(KS), arr(has_res), arr(accum), arr(rows)
    cap = 200000
    items, off, bal = np.zeros((cap, 5), np.int32), np.zeros(grid + 1, np.int32), ctypes.c_double()
    cnt = _native.check(lib.svb_tc_schedule_probe_ragged(n, ks.ctypes.data, hr.ctypes.data, ac.ctypes.data, Cin, len(rows),
                                                         rw.ctypes.data, MT, col_blocks, int(chain_ordered), grid, items.ctypes.data,
                                                         cap, off.ctypes.data, ctypes.byref(bal)), 'tc_schedule_probe_ragged')
    return items[:cnt], off, bal.value


ROWS = (np.random.RandomState(1234).randint(86, 1379, 16) * 8).tolist()      # stage 0 of the 1-16 s benchmark batch


@pytest.mark.parametrize('MT', [1, 2])
@pytest.mark.parametrize('col_blocks', [1, 2])
def test_ragged_schedule_covers_each_clips_tiles_once(lib, MT, col_blocks):
    rows = ROWS + [1, 127, 128, 129]
    items, off, bal = _schedule(lib, [3, 7, 11], [0, 0, 0], [0, 0, 0], rows, MT, col_blocks, False)
    assert off[0] == 0 and off[-1] == len(items) and (np.diff(off) <= 120).all()
    want = set()
    for l in range(3):
        for nb in range(col_blocks):
            for b, r in enumerate(rows):
                want |= {(l, nb, b, t) for t in range(-(-r // 128))}
    got = []
    for l, nb, b, t0, mt in items:
        assert t0 % 128 == 0 and t0 < rows[b], (b, t0, rows[b])          # nothing starts at or past the clip's end
        assert 1 <= mt <= MT and t0 + (mt - 1) * 128 < rows[b]              # nor covers a tile wholly past it
        got += [(l, nb, b, t0 // 128 + i) for i in range(mt)]
    assert len(got) == len(set(got)) and set(got) == want
    print(f'MT {MT} col_blocks {col_blocks}: {len(items)} items, balance {bal:.3f}')
    assert 0.5 < bal <= 1.0


def test_ragged_chain_ordered_schedule_keeps_a_tiles_layers_together(lib):
    rows = [300, 1, 129, 1000, 64]
    items, off, bal = _schedule(lib, [3, 7, 11], [1, 1, 1], [0, 1, 1], rows, 2, 2, True, grid=16, Cin=256)
    tiles = [(r + 127) // 128 for r in rows]
    assert len(items) == 3 * 2 * sum((t + 1) // 2 for t in tiles)
    for c in range(len(off) - 1):
        mine = items[off[c]:off[c + 1]]
        assert len(mine) % 3 == 0
        for i in range(0, len(mine), 3):
            assert mine[i:i + 3, 0].tolist() == [0, 1, 2]
            assert (mine[i:i + 3, 1:] == mine[i, 1:]).all()
    print(f'chain-ordered: balance {bal:.3f}')


def test_uniform_rows_give_the_uniform_schedule(lib):
    from tests.test_native_abi import _schedule as uniform
    a, oa, ba = uniform([3, 7, 11], [0, 0, 0], [0, 0, 0], 4, 1000, 2, 1, False)
    b, ob, bb = _schedule(lib, [3, 7, 11], [0, 0, 0], [0, 0, 0], [1000] * 4, 2, 1, False)
    assert np.array_equal(a, b) and np.array_equal(oa, ob) and ba == bb


def test_ragged_entry_points_validate_arguments_without_gpu(lib):
    """Rejected before any CUDA call (negative svb_status, message set)."""
    u64 = ctypes.c_uint64(1)
    i32 = lambda v: np.ascontiguousarray(v, dtype=np.int32)
    good, zero, long_ = i32([3, 5]), i32([3, 0]), i32([3, 9])
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    fwd = lambda lens, T_max: lib.svb_gen_forward_ragged(None, None, None, lens, None, None, u64, 2, T_max, None, None)
    assert fwd(None, 8) < 0 and b'lengths is NULL' in lib.svb_last_error()
    assert fwd(p(zero), 8) < 0 and b'outside [1, T_max 8]' in lib.svb_last_error()
    assert fwd(p(long_), 8) < 0 and b'length 9 of clip 1' in lib.svb_last_error()
    assert fwd(p(good), 8) < 0 and b'null handle' in lib.svb_last_error()
    assert fwd(p(good), 0) < 0 and b'T_max 0' in lib.svb_last_error()
    mel = np.zeros((8, 80), np.float32)
    out = np.zeros(8 * 256, np.float32)
    host = lambda lens: lib.svb_gen_spec2wav_ragged_host(None, p(mel), None, lens, 2, u64, p(out), None)
    assert host(None) < 0 and b'lengths is NULL' in lib.svb_last_error()
    assert host(p(zero)) < 0 and b'length 0 of clip 1' in lib.svb_last_error()
    assert host(p(good)) < 0 and b'not finalized' in lib.svb_last_error()
    assert lib.svb_gen_spec2wav_ragged_host(None, None, None, p(good), 2, u64, p(out), None) < 0 and b'null buffer' in lib.svb_last_error()
    q = np.zeros(8 * 256, np.int16)
    assert lib.svb_gen_spec2wav_ragged_host_i16(None, p(mel), None, p(zero), 2, u64, 1, p(q), None) < 0
    assert b'spec2wav_ragged_i16' in lib.svb_last_error()
    rows = i32([5, 0])
    ks = i32([3])
    assert lib.svb_tc_schedule_probe_ragged(1, p(ks), p(i32([0])), p(i32([0])), 128, 2, p(rows), 2, 1, 0, 8, p(np.zeros(100, np.int32)),
                                            20, p(np.zeros(9, np.int32)), ctypes.byref(ctypes.c_double())) < 0
    assert b'clip 1 has 0 rows' in lib.svb_last_error()


def test_binding_covers_the_ragged_entry_points():
    declared = set(_native.declared_symbols())
    for name in ('svb_gen_forward_ragged', 'svb_gen_spec2wav_ragged_host', 'svb_gen_spec2wav_ragged_host_i16',
                 'svb_tc_schedule_probe_ragged'):
        assert name in declared and name in _native._PROTOS
