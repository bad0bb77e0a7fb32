"""Host-side mirror of the reference generator interface, backed by libsvb_vocoder.so.

``HifiGanGenerator(h, c_out=1)`` keeps the reference's constructor, parameter /
state_dict names (so ``load_state_dict(ckpt['state_dict']['model_gen'],
strict=True)`` works on reference checkpoints), ``remove_weight_norm()`` and
``forward(x, f0=None)`` (reference: modules/hifigan/hifigan.py:104-178).  The
modules below are parameter containers only -- there is no PyTorch compute
path: ``forward`` hands raw device pointers to ``svb_gen_forward`` and raises
if the CUDA library or a CUDA device is missing.
"""
import ctypes

import numpy as np
import torch
from torch import nn

from neuralsvb_b200 import _native

LRELU_SLOPE = 0.1


def get_padding(kernel_size, dilation=1):
    return (kernel_size * dilation - dilation) // 2


class _WNConv(nn.Module):
    """Parameters of a weight-normalised conv: ``bias``, ``weight_g``, ``weight_v``
    (the names torch.nn.utils.weight_norm registers; hifigan.py:35-50,118,124,140).
    After ``fold()`` it holds ``bias`` and ``weight`` like remove_weight_norm leaves it."""

    def __init__(self, shape, n_bias, std=0.01):
        super().__init__()
        v = torch.randn(*shape) * std
        self.bias = nn.Parameter(torch.zeros(n_bias))
        self.weight_g = nn.Parameter(v.flatten(1).norm(dim=1).view(-1, *([1] * (len(shape) - 1))))
        self.weight_v = nn.Parameter(v)

    @property
    def folded(self):
        return 'weight' in self._parameters

    def effective_weight(self):
        """g * v / ||v|| (norm over all dims but 0), computed by the device kernel."""
        if self.folded:
            return self.weight.detach()
        v = self.weight_v.detach().float().cpu().contiguous()
        g = self.weight_g.detach().float().cpu().contiguous().view(-1)
        w = torch.empty_like(v)
        lib = _native.lib()
        dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
        _native.check(lib.svb_fold_weight_norm_host(_native.ptr(v), _native.ptr(g), v.shape[0], v[0].numel(),
                                                    _native.ptr(w), dev), 'fold_weight_norm')
        return w

    def fold(self):
        if self.folded:
            return
        w = self.effective_weight().to(self.weight_v.device)
        del self._parameters['weight_g'], self._parameters['weight_v']
        self.weight = nn.Parameter(w)


class _PlainConv(nn.Module):
    def __init__(self, shape, n_bias):
        super().__init__()
        bound = 1.0 / np.sqrt(np.prod(shape[1:]))
        self.weight = nn.Parameter(torch.empty(*shape).uniform_(-bound, bound))
        self.bias = nn.Parameter(torch.empty(n_bias).uniform_(-bound, bound))


class _GenTrainFn(torch.autograd.Function):
    """Autograd node of one training forward of the native generator (replaces torch autograd through
    hifigan.py:144-169).  Inputs after ``seed`` are the parameters, in ``_param_entries`` order."""

    @staticmethod
    def forward(ctx, gen, x, f0, rand_ini, noise, seed, *params):
        ctx.gen = gen
        ctx.n_params = len(params)
        return gen._run_forward(x, f0, rand_ini, noise, seed, train=True)

    @staticmethod
    def backward(ctx, dy):
        grads = ctx.gen._native_backward(dy)
        assert len(grads) == ctx.n_params
        return (None, None, None, None, None, None) + tuple(grads)


class ResBlock1(nn.Module):
    """Parameter container for hifigan.py:30-67."""

    def __init__(self, h, channels, kernel_size=3, dilation=(1, 3, 5)):
        super().__init__()
        self.h, self.kernel_size, self.dilation = h, kernel_size, tuple(dilation)
        self.convs1 = nn.ModuleList([_WNConv((channels, channels, kernel_size), channels) for _ in dilation])
        self.convs2 = nn.ModuleList([_WNConv((channels, channels, kernel_size), channels) for _ in dilation])

    def remove_weight_norm(self):
        for l in list(self.convs1) + list(self.convs2):
            l.fold()


class ResBlock2(nn.Module):
    """Parameter container for hifigan.py:70-91."""

    def __init__(self, h, channels, kernel_size=3, dilation=(1, 3)):
        super().__init__()
        self.h, self.kernel_size, self.dilation = h, kernel_size, tuple(dilation)
        self.convs = nn.ModuleList([_WNConv((channels, channels, kernel_size), channels) for _ in dilation])

    def remove_weight_norm(self):
        for l in self.convs:
            l.fold()


class _SourceModule(nn.Module):
    """m_source: only ``l_linear`` carries parameters (source.py:371-379)."""

    def __init__(self, harmonic_num):
        super().__init__()
        self.l_linear = nn.Linear(harmonic_num + 1, 1)


class HifiGanGenerator(nn.Module):
    def __init__(self, h, c_out=1, precision=None):
        super().__init__()
        if c_out != 1:
            raise ValueError('the CUDA generator implements c_out=1 (the only value the reference uses)')
        self.h = h
        self.num_kernels = len(h['resblock_kernel_sizes'])
        self.num_upsamples = len(h['upsample_rates'])
        self.precision = precision or h.get('svb_precision', 'bf16x3')
        self.n_mel = int(h.get('audio_num_mel_bins', 80))
        c0 = h['upsample_initial_channel']
        if h['use_pitch_embed']:
            self.harmonic_num = 8
            self.m_source = _SourceModule(self.harmonic_num)
            self.noise_convs = nn.ModuleList()
        self.conv_pre = _WNConv((c0, self.n_mel, 7), c0)
        self.ups = nn.ModuleList()
        for i, (u, k) in enumerate(zip(h['upsample_rates'], h['upsample_kernel_sizes'])):
            c_cur = c0 // (2 ** (i + 1))
            self.ups.append(_WNConv((c_cur * 2, c_cur, k), c_cur))          # ConvTranspose1d: [Cin, Cout, K]
            if h['use_pitch_embed']:
                if i + 1 < len(h['upsample_rates']):
                    s = int(np.prod(h['upsample_rates'][i + 1:]))
                    self.noise_convs.append(_PlainConv((c_cur, 1, s * 2), c_cur))
                else:
                    self.noise_convs.append(_PlainConv((c_cur, 1, 1), c_cur))
        self.resblocks = nn.ModuleList()
        rb = ResBlock1 if h['resblock'] == '1' else ResBlock2
        for i in range(len(self.ups)):
            ch = c0 // (2 ** (i + 1))
            for k, d in zip(h['resblock_kernel_sizes'], h['resblock_dilation_sizes']):
                self.resblocks.append(rb(h, ch, k, d))
        self.conv_post = _WNConv((c_out, ch, 7), c_out)
        self._handle = None
        self._handle_key = None
        self._synced_version = None
        self.seed = 0

    # ------------------------------------------------------------------ reference API
    def remove_weight_norm(self):
        print('Removing weight norm...')
        for l in self.ups:
            l.fold()
        for l in self.resblocks:
            l.remove_weight_norm()
        self.conv_pre.fold()
        self.conv_post.fold()
        self._drop_handle()

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self._drop_handle()
        return r

    def forward(self, x, f0=None, rand_ini=None, noise=None, seed=None, lengths=None):
        """x [B, n_mel, T] fp32 on a CUDA device, f0 [B, T] Hz or None -> [B, 1, T*hop].
        ``rand_ini`` [B,9] / ``noise`` [B,T*hop,9] inject the NSF source's random draws
        (parity testing); otherwise they are drawn in-kernel from ``seed``.

        ``lengths`` (list, or CPU / CUDA integer tensor [B], 1 <= lengths[b] <= T): a ragged batch in one launch
        sequence (svb_gen_forward_ragged).  Clip b's first ``lengths[b]*hop`` samples equal a forward of
        ``x[b:b+1, :, :lengths[b]]`` alone (same injected noise); the rest of its row is 0 and nothing of ``x`` / ``f0`` /
        ``noise`` past its length is read.  The schedule is built on the host, so a CUDA tensor costs one device-to-host
        copy (and a sync).  Inference only: with grad in ``train()`` mode it raises ``NotImplementedError``.

        In ``train()`` mode with grad enabled the result carries a grad_fn: ``backward`` runs
        ``svb_gen_backward`` (native data / weight gradients) and hands every parameter its gradient
        (weight-norm ``weight_g`` / ``weight_v`` through ``svb_weight_norm_backward``)."""
        if not x.is_cuda:
            raise RuntimeError('HifiGanGenerator.forward needs CUDA tensors: there is no CPU fallback '
                               '(the reference CPU path lives in the oracle, for tests only)')
        train = self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if seed is None:
            self.seed += 1
            seed = self.seed
        if train:
            if lengths is not None:
                raise NotImplementedError('ragged batches (lengths=...) are inference only: the training tape takes clips of equal length')
            entries = self._param_entries()
            return _GenTrainFn.apply(self, x, f0, rand_ini, noise, seed, *[p for e in entries for p in e[2]])
        return self._run_forward(x, f0, rand_ini, noise, seed, train=False, lengths=lengths)

    def _run_forward(self, x, f0, rand_ini, noise, seed, train, lengths=None):
        lib = _native.lib()
        g = self._ensure_handle(x.device)
        g = self._sync_weights(g, train)
        B, C, T = x.shape
        if C != self.n_mel:
            raise ValueError(f'expected {self.n_mel} mel bins, got {C}')
        x = x.contiguous().float()
        f0 = None if f0 is None else f0.contiguous().float().to(x.device)
        hop = int(lib.svb_gen_hop(g))
        y = torch.empty(B, 1, T * hop, device=x.device, dtype=torch.float32)
        ri = None if rand_ini is None else rand_ini.contiguous().float().to(x.device)
        nz = None if noise is None else noise.contiguous().float().to(x.device)
        if lengths is not None:
            if torch.is_tensor(lengths):
                lengths = lengths.detach().to('cpu')           # the one device-to-host copy of a CUDA tensor
            lens = np.ascontiguousarray(np.asarray(lengths).reshape(-1), dtype=np.int64)
            if lens.shape != (B,):
                raise ValueError(f'lengths has {lens.size} entries for a batch of {B}')
            if (lens < 1).any() or (lens > T).any():
                raise ValueError(f'lengths must lie in [1, {T}], got {lens.tolist()}')
            lens = lens.astype(np.int32)
        with torch.cuda.device(x.device):
            st = _native.current_stream_ptr(x.device)
            if lengths is None:
                _native.check(lib.svb_gen_forward(g, _native.ptr(x), _native.ptr(f0), _native.ptr(ri), _native.ptr(nz),
                                                  ctypes.c_uint64(seed), B, T, _native.ptr(y), st), 'gen_forward')
            else:
                _native.check(lib.svb_gen_forward_ragged(g, _native.ptr(x), _native.ptr(f0), lens.ctypes.data_as(ctypes.c_void_p),
                                                         _native.ptr(ri), _native.ptr(nz), ctypes.c_uint64(seed), B, T,
                                                         _native.ptr(y), st), 'gen_forward_ragged')
        return y

    # ------------------------------------------------------------------ training
    def _param_entries(self):
        """[(reference prefix, module, [parameters in the order backward returns their gradients])]"""
        out = []

        def put(prefix, m):
            ps = [m.bias, m.weight] if (isinstance(m, _PlainConv) or m.folded) else [m.bias, m.weight_g, m.weight_v]
            out.append((prefix, m, ps))
        put('conv_pre', self.conv_pre)
        put('conv_post', self.conv_post)
        for i, l in enumerate(self.ups):
            put(f'ups.{i}', l)
        for n, rb in enumerate(self.resblocks):
            for attr in (('convs1', 'convs2') if isinstance(rb, ResBlock1) else ('convs',)):
                for m, l in enumerate(getattr(rb, attr)):
                    put(f'resblocks.{n}.{attr}.{m}', l)
        if self.h['use_pitch_embed']:
            for i, l in enumerate(self.noise_convs):
                put(f'noise_convs.{i}', l)
            out.append(('m_source.l_linear', self.m_source.l_linear, [self.m_source.l_linear.bias, self.m_source.l_linear.weight]))
        return out

    def _sync_weights(self, g, train):
        """Keep the native packings in step with the parameters (they change after every optimizer step)."""
        lib = _native.lib()
        _native.check(lib.svb_gen_set_training(g, 1 if train else 0), 'set_training')
        ver = tuple(p._version for p in self.parameters())
        if ver == self._synced_version:
            return g
        if not train:                                   # inference handle: rebuild from scratch
            dev = torch.device('cuda', self._handle_key)
            self._drop_handle()
            return self._ensure_handle(dev)
        # device-side: fold weight norm, hand every folded tensor over, rebuild all packings with gather / tile kernels
        dev = torch.device('cuda', self._handle_key)
        with torch.cuda.device(dev):
            st = _native.current_stream_ptr(dev)

            def put(name, t):
                t = t.detach()
                if t.dtype != torch.float32 or not t.is_contiguous():
                    t = t.float().contiguous()
                _native.check(lib.svb_gen_set_weight_dev(g, name.encode(), _native.ptr(t), t.numel(), st), f'set_weight_dev({name})')
            for prefix, m, ps in self._param_entries():
                put(prefix + '.bias', ps[0])
                if len(ps) == 2:
                    put(prefix + '.weight', ps[1])
                    continue
                v, gv = m.weight_v.detach(), m.weight_g.detach()
                if getattr(m, '_w_scratch', None) is None or m._w_scratch.shape != v.shape or m._w_scratch.device != v.device:
                    m._w_scratch = torch.empty_like(v, dtype=torch.float32)
                _native.check(lib.svb_fold_weight_norm_dev(_native.ptr(v), _native.ptr(gv), v.shape[0], v[0].numel(),
                                                           _native.ptr(m._w_scratch), st), 'fold_weight_norm_dev')
                put(prefix + '.weight', m._w_scratch)
            _native.check(lib.svb_gen_update_weights_dev(g, st), 'update_weights_dev')
        self._synced_version = ver
        return g

    def _native_backward(self, dy):
        """d(loss)/d(wav) [B,1,T*hop] -> flat list of parameter gradients in ``_param_entries`` order."""
        lib = _native.lib()
        g = self._handle
        dev = dy.device
        dy = dy.contiguous().float()
        grads = []
        with torch.cuda.device(dev):
            st = _native.current_stream_ptr(dev)
            _native.check(lib.svb_gen_zero_grad(g, st), 'zero_grad')
            _native.check(lib.svb_gen_backward(g, _native.ptr(dy), st), 'gen_backward')

            def fetch(name, like):
                n = int(lib.svb_gen_grad_numel(g, name.encode()))
                if n != like.numel():
                    raise RuntimeError(f'gradient {name}: native {n} elements, parameter {like.numel()}')
                t = torch.empty(like.shape, device=dev, dtype=torch.float32)
                _native.check(lib.svb_gen_get_grad(g, name.encode(), _native.ptr(t), n, st), f'get_grad({name})')
                return t
            for prefix, m, ps in self._param_entries():
                db = fetch(prefix + '.bias', ps[0])
                if len(ps) == 2:
                    grads += [db, fetch(prefix + '.weight', ps[1])]
                    continue
                v = m.weight_v.detach().float().contiguous()
                gv = m.weight_g.detach().float().contiguous()
                dw = fetch(prefix + '.weight', v)
                dv, dg = torch.empty_like(v), torch.empty_like(gv)
                _native.check(lib.svb_weight_norm_backward(_native.ptr(v), _native.ptr(gv), _native.ptr(dw), v.shape[0],
                                                           v[0].numel(), _native.ptr(dv), _native.ptr(dg), st),
                              'weight_norm_backward')
                grads += [db, dg, dv]
        return grads

    # ------------------------------------------------------------------ native handle
    def folded_state(self):
        """{reference name: folded fp32 CPU tensor} for every tensor the kernels need."""
        out = {}

        def put(prefix, m):
            out[prefix + '.weight'] = m.effective_weight().float().cpu().contiguous()
            out[prefix + '.bias'] = m.bias.detach().float().cpu().contiguous()
        put('conv_pre', self.conv_pre)
        put('conv_post', self.conv_post)
        for i, l in enumerate(self.ups):
            put(f'ups.{i}', l)
        for n, rb in enumerate(self.resblocks):
            if isinstance(rb, ResBlock1):
                for m, l in enumerate(rb.convs1):
                    put(f'resblocks.{n}.convs1.{m}', l)
                for m, l in enumerate(rb.convs2):
                    put(f'resblocks.{n}.convs2.{m}', l)
            else:
                for m, l in enumerate(rb.convs):
                    put(f'resblocks.{n}.convs.{m}', l)
        if self.h['use_pitch_embed']:
            for i, l in enumerate(self.noise_convs):
                out[f'noise_convs.{i}.weight'] = l.weight.detach().float().cpu().contiguous()
                out[f'noise_convs.{i}.bias'] = l.bias.detach().float().cpu().contiguous()
            out['m_source.l_linear.weight'] = self.m_source.l_linear.weight.detach().float().cpu().contiguous()
            out['m_source.l_linear.bias'] = self.m_source.l_linear.bias.detach().float().cpu().contiguous()
        return out

    def native_config(self):
        h = self.h
        c = _native.GenConfig()
        c.n_mel = self.n_mel
        c.upsample_initial_channel = h['upsample_initial_channel']
        c.n_ups = len(h['upsample_rates'])
        for i, (u, k) in enumerate(zip(h['upsample_rates'], h['upsample_kernel_sizes'])):
            c.upsample_rates[i], c.upsample_kernel_sizes[i] = int(u), int(k)
        c.resblock = 1 if h['resblock'] == '1' else 2
        c.n_resblock_kernels = len(h['resblock_kernel_sizes'])
        nd = len(h['resblock_dilation_sizes'][0])
        c.n_dilations = nd
        for j, (k, d) in enumerate(zip(h['resblock_kernel_sizes'], h['resblock_dilation_sizes'])):
            c.resblock_kernel_sizes[j] = int(k)
            if len(d) != nd:
                raise ValueError('all ResBlocks must have the same number of dilations')
            for m, dd in enumerate(d):
                c.resblock_dilation_sizes[j][m] = int(dd)
        c.use_pitch_embed = 1 if h['use_pitch_embed'] else 0
        c.audio_sample_rate = int(h['audio_sample_rate'])
        c.precision = _native.PREC[self.precision]
        return c

    def set_precision(self, precision):
        self.precision = precision
        if self._handle is not None:
            _native.check(_native.lib().svb_gen_set_precision(self._handle, _native.PREC[precision]), 'set_precision')

    def _drop_handle(self):
        if getattr(self, '_handle', None) is not None:
            _native.lib().svb_gen_destroy(self._handle)
        self._handle, self._handle_key = None, None

    def _ensure_handle(self, device):
        key = (device.index if device.index is not None else torch.cuda.current_device())
        if self._handle is not None and self._handle_key == key:
            return self._handle
        self._drop_handle()
        lib = _native.lib()
        cfg = self.native_config()
        hnd = ctypes.c_void_p()
        _native.check(lib.svb_gen_create(ctypes.byref(cfg), key, ctypes.byref(hnd)), 'gen_create')
        try:
            for name, t in self.folded_state().items():
                shape = (ctypes.c_int64 * t.dim())(*t.shape)
                _native.check(lib.svb_gen_set_weight(hnd, name.encode(), _native.ptr(t), shape, t.dim()),
                              f'set_weight({name})')
            _native.check(lib.svb_gen_finalize(hnd), 'gen_finalize')
        except Exception:
            lib.svb_gen_destroy(hnd)
            raise
        self._handle, self._handle_key = hnd, key
        self._synced_version = tuple(p._version for p in self.parameters())
        return hnd

    def native_handle(self, device=None):
        device = device or torch.device('cuda', torch.cuda.current_device())
        return self._ensure_handle(device)

    def get_tap(self, name, device=None):
        """Named activation of the last forward as [B, C, T] (layer-level parity tests)."""
        lib = _native.lib()
        g = self._handle
        dev = torch.device('cuda', self._handle_key)
        cap = 1 << 28
        shape = (ctypes.c_int64 * 3)()
        # query size first with a generous scratch buffer sized from the output
        buf = torch.empty(cap // 4, device=dev, dtype=torch.float32)
        _native.check(lib.svb_gen_get_tap(g, name.encode(), _native.ptr(buf), buf.numel(), shape,
                                          _native.current_stream_ptr(dev)), f'get_tap({name})')
        B, C, T = shape[0], shape[1], shape[2]
        return buf[:B * C * T].view(B, C, T).clone()

    def __del__(self):
        try:
            self._drop_handle()
        except Exception:
            pass
