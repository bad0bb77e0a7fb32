"""ctypes binding of libsvb_vocoder.so (C ABI declared in include/svb_vocoder.h).

The library is built in-tree by ``build()`` (nvcc, sm_100a only) and loaded by
``lib()``.  There is no CPU or PyTorch fallback anywhere in this package: if the
library is missing, or a call fails, a ``RuntimeError`` is raised.
"""
import ctypes
import os
import shutil
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, 'csrc')
LIB_PATH = os.path.join(_HERE, 'libsvb_vocoder.so')
HEADER = os.path.join(_ROOT, 'include', 'svb_vocoder.h')
SOURCES = ['wn.cu', 'conformer.cu', 'api.cu', 'conv_ffma.cu', 'conv_tc.cu', 'nsf_source.cu', 'frontend.cu', 'generator.cu', 'layer_api.cu', 'disc_ops.cu',
           'train_ops.cu', 'generator_bwd.cu', 'disc_bwd.cu', 'tc_layer.cu', 'wgrad_tc.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared']

SVB_MAX_UPS, SVB_MAX_RBK, SVB_MAX_DIL = 8, 4, 4
PREC = {'fp32': 0, 'tf32': 1, 'tf32x3': 2, 'bf16x3': 3}
PAD_CENTER_ZERO, PAD_CENTER_REFLECT, PAD_HALF_REFLECT = 0, 1, 2
OUT_LOG10_MEL, OUT_LN_MEL, OUT_MAG, OUT_MAG_RAW, OUT_MEL_MAG = 0, 1, 2, 3, 4


class GenConfig(ctypes.Structure):
    _fields_ = [
        ('n_mel', ctypes.c_int32),
        ('upsample_initial_channel', ctypes.c_int32),
        ('n_ups', ctypes.c_int32),
        ('upsample_rates', ctypes.c_int32 * SVB_MAX_UPS),
        ('upsample_kernel_sizes', ctypes.c_int32 * SVB_MAX_UPS),
        ('resblock', ctypes.c_int32),
        ('n_resblock_kernels', ctypes.c_int32),
        ('resblock_kernel_sizes', ctypes.c_int32 * SVB_MAX_RBK),
        ('n_dilations', ctypes.c_int32),
        ('resblock_dilation_sizes', (ctypes.c_int32 * SVB_MAX_DIL) * SVB_MAX_RBK),
        ('use_pitch_embed', ctypes.c_int32),
        ('audio_sample_rate', ctypes.c_int32),
        ('precision', ctypes.c_int32),
    ]


class StftConfig(ctypes.Structure):
    _fields_ = [
        ('n_fft', ctypes.c_int32), ('hop', ctypes.c_int32), ('win', ctypes.c_int32),
        ('pad_mode', ctypes.c_int32), ('out_kind', ctypes.c_int32), ('clamp_input', ctypes.c_int32),
        ('n_mels', ctypes.c_int32), ('frames_major', ctypes.c_int32), ('eps', ctypes.c_float),
    ]


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + [HEADER] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source into neuralsvb_b200/libsvb_vocoder.so for sm_100a."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        raise RuntimeError('nvcc not found: cannot build libsvb_vocoder.so')
    cmd = [nvcc] + NVCC_FLAGS + sources() + ['-o', LIB_PATH + '.tmp']
    if verbose:
        print(' '.join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + r.stdout + r.stderr)
    os.replace(LIB_PATH + '.tmp', LIB_PATH)
    return LIB_PATH


_lib = None
_lock = threading.Lock()

_P = ctypes.c_void_p
_I32, _I64, _U64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64

_PROTOS = {
    # name: (restype, argtypes)
    'svb_last_error': (ctypes.c_char_p, []),
    'svb_abi_version': (ctypes.c_int, []),
    'svb_gen_create': (ctypes.c_int, [ctypes.POINTER(GenConfig), ctypes.c_int, ctypes.POINTER(_P)]),
    'svb_gen_destroy': (None, [_P]),
    'svb_gen_set_weight': (ctypes.c_int, [_P, ctypes.c_char_p, _P, ctypes.POINTER(_I64), _I32]),
    'svb_fold_weight_norm_host': (ctypes.c_int, [_P, _P, _I64, _I64, _P, ctypes.c_int]),
    'svb_gen_finalize': (ctypes.c_int, [_P]),
    'svb_gen_set_precision': (ctypes.c_int, [_P, _I32]),
    'svb_gen_forward': (ctypes.c_int, [_P, _P, _P, _P, _P, _U64, _I32, _I32, _P, _P]),
    'svb_gen_spec2wav_host': (ctypes.c_int, [_P, _P, _P, _U64, _I32, _I32, _P, _P]),
    'svb_gen_get_tap': (ctypes.c_int, [_P, ctypes.c_char_p, _P, _I64, ctypes.POINTER(_I64), _P]),
    'svb_gen_hop': (_I64, [_P]),
    'svb_gen_last_launches': (_I64, [_P]),
    'svb_gen_last_flops': (ctypes.c_double, [_P]),
    'svb_gen_enable_timing': (ctypes.c_int, [_P, _I32]),
    'svb_gen_last_ms': (ctypes.c_float, [_P]),
    'svb_conv_nct_backward': (ctypes.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32,
                                             ctypes.c_float, _P, _P, _P, _P, _P]),
    'svb_avgpool1d_4_2_1_backward': (ctypes.c_int, [_P, _P, _I64, _I32, _P]),
    'svb_cond_net_forward': (ctypes.c_int, [_P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P]),
    'svb_cond_net_backward': (ctypes.c_int, [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P, _P]),
    'svb_pad_reflect_right_backward': (ctypes.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    'svb_loss_grad': (ctypes.c_int, [_P, _P, _I32, ctypes.c_float, _P, _I64, _I32, _P]),
    'svb_loss_grad_dev': (ctypes.c_int, [_P, _P, _I32, ctypes.c_float, _P, _P, _I64, _I32, _P]),
    'svb_tc_layer_create': (ctypes.c_int, [_I32, _I32, _I32, _I32, _I32, _I32, ctypes.c_int, ctypes.POINTER(_P)]),
    'svb_tc_layer_create_grouped': (ctypes.c_int, [_I32, _I32, _I32, _I32, _I32, _I32, _I32, ctypes.c_int, ctypes.POINTER(_P)]),
    'svb_tc_layer_destroy': (None, [_P]),
    'svb_tc_layer_set_weight_dev': (ctypes.c_int, [_P, _P, _P, _P]),
    'svb_tc_layer_out_len': (_I64, [_P, _I64]),
    'svb_tc_layer_forward': (ctypes.c_int, [_P, _P, _I32, _I32, _I32, ctypes.c_float, _P, _P]),
    'svb_tc_layer_backward': (ctypes.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, ctypes.c_float, _P, _P, _P, _P]),
    'svb_gen_set_training': (ctypes.c_int, [_P, _I32]),
    'svb_gen_update_weights': (ctypes.c_int, [_P]),
    'svb_gen_zero_grad': (ctypes.c_int, [_P, _P]),
    'svb_gen_set_weight_dev': (ctypes.c_int, [_P, ctypes.c_char_p, _P, _I64, _P]),
    'svb_gen_update_weights_dev': (ctypes.c_int, [_P, _P]),
    'svb_fold_weight_norm_dev': (ctypes.c_int, [_P, _P, _I64, _I64, _P, _P]),
    'svb_gen_backward': (ctypes.c_int, [_P, _P, _P]),
    'svb_gen_grad_numel': (_I64, [_P, ctypes.c_char_p]),
    'svb_gen_get_grad': (ctypes.c_int, [_P, ctypes.c_char_p, _P, _I64, _P]),
    'svb_gen_bwd_launches': (_I64, [_P]),
    'svb_weight_norm_backward': (ctypes.c_int, [_P, _P, _P, _I64, _I64, _P, _P, _P]),
    'svb_gen_profile_count': (_I32, [_P]),
    'svb_gen_profile_get': (ctypes.c_int, [_P, _I32, ctypes.c_char_p, _I32, ctypes.POINTER(ctypes.c_float),
                                            ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    'svb_conv1d_run': (ctypes.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, ctypes.c_float,
                                      ctypes.c_float, _I32, _I32, _P, ctypes.POINTER(ctypes.c_float), _P]),
    'svb_conv_nct_forward': (ctypes.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32,
                                            ctypes.c_float, _P]),
    'svb_avgpool1d_4_2_1': (ctypes.c_int, [_P, _P, _I64, _I32, _P]),
    'svb_pad_reflect_right': (ctypes.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    'svb_pair_stats': (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P]),
    'svb_spectral_sigma_host': (ctypes.c_int, [_P, _P, _P, _I64, _I64, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]),
    'svb_stft_num_frames': (_I64, [ctypes.POINTER(StftConfig), _I64]),
    'svb_stft_forward': (ctypes.c_int, [ctypes.POINTER(StftConfig), _P, _I32, _I64, _P, _P, _P]),
    'svb_stft_backward': (ctypes.c_int, [ctypes.POINTER(StftConfig), _P, _I32, _I64, _P, _P, _P, _P]),
    'svb_denoise': (ctypes.c_int, [ctypes.POINTER(StftConfig), _P, _I32, _I64, ctypes.c_float, _P, _P]),
    'svb_wav2spec_host': (_I64, [ctypes.POINTER(StftConfig), _P, _I64, _P, _P, _P, ctypes.c_int, _P]),
    'svb_wav2spec_batch_host': (_I64, [ctypes.POINTER(StftConfig), _P, _P, _I32, _P, _P, _P, ctypes.c_int, _P]),
    'svb_gen_spec2wav_host_i16': (ctypes.c_int, [_P, _P, _P, _U64, _I32, _I32, _I32, _P, _P]),
    'svb_wav_to_int16': (ctypes.c_int, [_P, _I32, _I64, _I32, _P, _P]),
    'svb_wn_create': (ctypes.c_int, [_I32, _I32, _I32, _I32, _I32, _I32, _I32, ctypes.POINTER(_P)]),
    'svb_wn_destroy': (None, [_P]),
    'svb_wn_set_weight': (ctypes.c_int, [_P, ctypes.c_char_p, _P, ctypes.POINTER(_I64), _I32]),
    'svb_wn_finalize': (ctypes.c_int, [_P]),
    'svb_wn_forward': (ctypes.c_int, [_P, _P, _P, _P, _I32, _I32, _P, _P]),
    'svb_fvae_decoder_create': (ctypes.c_int, [_I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, ctypes.POINTER(_P)]),
    'svb_fvae_decoder_forward': (ctypes.c_int, [_P, _P, _P, _P, _I32, _I32, _P, _P]),
    'svb_tc_schedule_probe': (_I64, [_I32, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _I64, _P, ctypes.POINTER(ctypes.c_double)]),
    'svb_tc_schedule_probe_ragged': (_I64, [_I32, _P, _P, _P, _I32, _I32, _P, _I32, _I32, _I32, _I32, _P, _I64, _P,
                                            ctypes.POINTER(ctypes.c_double)]),
    'svb_gen_forward_ragged': (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _U64, _I32, _I32, _P, _P]),
    'svb_gen_spec2wav_ragged_host': (ctypes.c_int, [_P, _P, _P, _P, _I32, _U64, _P, _P]),
    'svb_gen_spec2wav_ragged_host_i16': (ctypes.c_int, [_P, _P, _P, _P, _I32, _U64, _I32, _P, _P]),
    'svb_layer_norm_nct': (ctypes.c_int, [_P, _P, _P, _I32, _I32, _I32, ctypes.c_float, _P, _P]),
    'svb_relpos_attention_nct': (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P, _P]),
}


def declared_symbols():
    """Every entry point include/svb_vocoder.h declares (parsed from the header)."""
    import re
    txt = open(HEADER).read()
    txt = re.sub(r'/\*.*?\*/', '', txt, flags=re.S)
    return sorted(set(re.findall(r'\b(svb_[a-z0-9_]+)\s*\(', txt)))


def lib():
    """The loaded library.  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                    '(nvcc, sm_100a). neuralsvb_b200 has no CPU or PyTorch fallback.')
            l = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in _PROTOS.items():
                if hasattr(l, name):
                    fn = getattr(l, name)
                    fn.restype, fn.argtypes = res, args
            _lib = l
    return _lib


def check(status, what=''):
    """Turn a negative svb_status into a RuntimeError carrying svb_last_error()."""
    if status is not None and status < 0:
        msg = lib().svb_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'libsvb_vocoder {what} failed ({status}): {msg}')
    return status


def ptr(t):
    """Device/host pointer of a contiguous fp32 torch tensor (or None)."""
    if t is None:
        return None
    assert t.is_contiguous(), 'native calls need contiguous tensors'
    return ctypes.c_void_p(t.data_ptr())


def current_stream_ptr(device=None):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
