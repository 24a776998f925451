"""Torch-facing wrappers over the C-ABI kernels (librw_b200.so).

Every function here takes CUDA fp32 tensors, allocates outputs with torch (the
library never allocates), and launches on torch's current stream.  Autograd is
provided by explicit `torch.autograd.Function`s whose backward passes are the
same tensor-core kernels run on gradient planes.

Reference call sites replaced (davidbau/rewriting): utils/stylegan2/models.py
313-329 (DemodulatedConv2dF), 535-546 (NoiseInjectionF), 616-626 (ApplyStyle,
FusedLeakyReLUF), 628-655 (ToRGBF), op/fused_act.py, op/upfirdn2d.py,
utils/runningstats.py:1086-1097, rewrite/ganrewrite.py:806-813.
"""
import ctypes
import math

import numpy as np
import torch

from . import _cabi


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t):
    """contiguous fp32 CUDA view of t (the reference ops call .contiguous() too:
    fused_bias_act_kernel.cu:58-60, upfirdn2d_kernel.cu:149-150)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise _cabi.RwError('rewriting_b200 ops need CUDA tensors (got %s); there is no CPU '
                            'fallback' % t.device)
    if t.dtype != torch.float32:
        raise _cabi.RwError('rewriting_b200 ops are fp32-in/fp32-out (got %s)' % t.dtype)
    return t.contiguous()


# --------------------------------------------------------------------------- noise
_NOISE_CACHE = {}


def noise_table(batch, hw, device, period=None):
    """The reference draws `np.random.RandomState(0).randn(batch, H*W)` on the host in
    every NoiseInjectionF.forward (models.py:542-545).  The values only depend on
    (batch, H*W); generate once and keep on the device.

    `period`: row i of the table is row (i % period) of `randn(period, H*W)` — what sample i of a
    stream gets when the reference processes it in batches of `period` (its tally loops use 10).
    Lets a large batch reproduce the reference's small-batch statistics exactly."""
    if period is not None and period >= batch:
        period = None
    key = (batch, hw, str(device), period)
    t = _NOISE_CACHE.get(key)
    if t is None:
        if period is None:
            arr = np.random.RandomState(0).randn(batch, hw).astype('float32')
        else:
            base = np.random.RandomState(0).randn(period, hw).astype('float32')
            arr = np.ascontiguousarray(base[np.arange(batch) % period])
        t = torch.from_numpy(arr).to(device)
        while len(_NOISE_CACHE) > 256:            # evict the oldest entry only; live CUDA graphs
            _NOISE_CACHE.pop(next(iter(_NOISE_CACHE)))   # keep their tables alive themselves
        _NOISE_CACHE[key] = t
    return t


def cached_device_state():
    """Every cached device tensor whose raw pointer a captured CUDA graph may have baked in
    (noise tables, weight planes, workspaces).  `GraphedModule` holds this list so that a cache
    eviction can never free memory a graph replay still reads."""
    return (list(_NOISE_CACHE.values()), [e[2] for e in _WEIGHT_CACHE.values()],
            list(_WS.values()))


# --------------------------------------------------------------------------- planes
class KeyPlanes(object):
    """bf16 hi/lo planes of a [B,C,H,W] tensor in the padded-flat channels-last layout."""
    __slots__ = ('hi', 'lo', 'B', 'C', 'H', 'W')

    def __init__(self, hi, lo, B, C, H, W):
        self.hi, self.lo, self.B, self.C, self.H, self.W = hi, lo, B, C, H, W

    @property
    def rows(self):
        return self.B * (self.H + 1) * (self.W + 1)


def prep_keys(x, scale_bc=None, want_k=False):
    """planes of (scale_bc[b,c] * x[b,c,y,x]); optionally also the fp32 NCHW product."""
    x = _f32c(x)
    scale_bc = _f32c(scale_bc)
    B, C, H, W = x.shape
    rows = B * (H + 1) * (W + 1)
    hi = torch.empty((rows, C), dtype=torch.bfloat16, device=x.device)
    lo = torch.empty_like(hi)
    k = torch.empty_like(x) if want_k else None
    _cabi.call('rw_prep_keys', _p(x), _p(scale_bc), B, C, H, W, _p(hi), _p(lo), _p(k), _stream())
    return KeyPlanes(hi, lo, B, C, H, W), k


def split_rows(a):
    a = _f32c(a)
    hi = torch.empty(a.shape, dtype=torch.bfloat16, device=a.device)
    lo = torch.empty_like(hi)
    _cabi.call('rw_split_rows', _p(a), a.numel(), _p(hi), _p(lo), _stream())
    return hi, lo


_WEIGHT_CACHE = {}


def weight_planes(weight, kind='fwd', scale=None):
    """(hi, lo, wsq) planes of scale*W for a [1,Cout,Cin,3,3] / [Cout,Cin,3,3] tensor.
    Cached per tensor OBJECT (weak reference) and `_version`: the rewriter mutates W in
    place, which bumps `_version` and invalidates the entry (SURVEY.md §8b); temporaries
    (e.g. linear_insert's W0 + Lambda d) are new objects and never hit a stale entry."""
    import weakref
    w = weight.detach()
    if w.dim() == 5:
        w = w[0]
    Cout, Cin, kh, kw = w.shape
    assert kh == 3 and kw == 3
    if scale is None:                  # StyleGAN2's equalised-lr factor (models.py:315-319)
        scale = 1.0 / math.sqrt(Cin * 9)
    key = (id(weight), kind, float(scale))
    ent = _WEIGHT_CACHE.get(key)
    if ent is not None and ent[0]() is weight and ent[1] == weight._version:
        return ent[2]
    w = _f32c(w)
    hi = torch.empty((Cout * 9 * Cin,), dtype=torch.bfloat16, device=w.device)
    lo = torch.empty_like(hi)
    if kind == 'fwd':
        wsq = torch.empty((Cout, Cin), dtype=torch.float32, device=w.device)
        _cabi.call('rw_prep_weights', _p(w), Cout, Cin, scale, 0, 0, _p(hi), _p(lo), _p(wsq),
                   _stream())
    elif kind == 'upf':        # [Cout/16][half][tap][8][Cin]: N = 144 tiles of the fused up-conv
        wsq = weight_planes(weight, 'fwd', scale)[2]
        _cabi.call('rw_prep_weights', _p(w), Cout, Cin, scale, 2, 0, _p(hi), _p(lo), None,
                   _stream())
    elif kind == 'dgrad':      # [Cin][flipped tap][Cout]
        wsq = None
        _cabi.call('rw_prep_weights', _p(w), Cout, Cin, scale, 1, 1, _p(hi), _p(lo), None,
                   _stream())
    elif kind == 'dgrad_up':   # [Cin][tap][Cout] (conv_transpose: taps are not flipped)
        wsq = None
        _cabi.call('rw_prep_weights', _p(w), Cout, Cin, scale, 1, 0, _p(hi), _p(lo), None,
                   _stream())
    else:
        raise ValueError(kind)
    val = (hi, lo, wsq)
    if isinstance(weight, torch.nn.Parameter):
        while len(_WEIGHT_CACHE) > 256:
            _WEIGHT_CACHE.pop(next(iter(_WEIGHT_CACHE)))
        _WEIGHT_CACHE[key] = (weakref.ref(weight), weight._version, val)
    return val


def rgb_parts(Cout):
    """Number of ToRGB partial sums rw_modconv_fwd_fused writes for a Cout-channel layer."""
    n = _cabi.load().rw_modconv_rgb_parts(int(Cout))
    if n < 1:
        raise _cabi.RwError('the row-GEMM does not take Cout=%d output channels' % Cout)
    return n


def demod_factors(style, wsq, eps=1e-8):
    style = _f32c(style)
    B, Cin = style.shape
    Cout = wsq.shape[0]
    out = torch.empty((B, Cout), dtype=torch.float32, device=style.device)
    _cabi.call('rw_demod', _p(style), _p(wsq), B, Cout, Cin, eps, _p(out), _stream())
    return out


_SEPARABLE = {}


def up_fused_eligible(Cin, Cout, H, W, blur_kernel):
    """Shapes the fused upsampling kernel takes (csrc/upconv_tc.cu): square power-of-two input of
    width 4..128, Cin % 64 == 0, Cout % 16 == 0, rank-one 4x4 FIR; RW_UP_FUSED=0 turns it off."""
    import os
    return (os.environ.get('RW_UP_FUSED', '1') != '0' and H == W and 4 <= W <= 128 and
            (W & (W - 1)) == 0 and Cin % 64 == 0 and Cout % 16 == 0 and
            tuple(blur_kernel.shape) == (4, 4) and blur_is_separable(blur_kernel))


def blur_is_separable(kernel):
    """True if the 4x4 FIR is rank one (the model's [1,3,3,1] x [1,3,3,1] always is), which the
    fused upsampling kernel requires.  One device->host read per kernel tensor version (done in
    the warm-up pass, never inside a graph capture)."""
    key = (kernel.data_ptr(), kernel._version, tuple(kernel.shape))
    r = _SEPARABLE.get(key)
    if r is None:
        k = kernel.detach().double().cpu()
        r = bool(tuple(k.shape) == (4, 4) and k[0, 0] != 0 and
                 torch.equal(k * k[0, 0], torch.outer(k[:, 0], k[0, :])))
        if len(_SEPARABLE) > 64:
            _SEPARABLE.clear()
        _SEPARABLE[key] = r
    return r


# --------------------------------------------------------------------------- conv kernels
def conv3x3_planes(planes, w_hi, w_lo, Cout, scale_bo=None, noise=None, noise_w=None, bias=None,
                   act=False):
    """row-GEMM 3x3 conv (pad 1) over key planes -> [B,Cout,H,W] fp32."""
    B, Cin, H, W = planes.B, planes.C, planes.H, planes.W
    out = torch.empty((B, Cout, H, W), dtype=torch.float32, device=planes.hi.device)
    nstride = noise.stride(0) if noise is not None else 0
    _cabi.call('rw_modconv_fwd', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo), _p(scale_bo),
               _p(noise), nstride, _p(noise_w), _p(bias), 1 if act else 0, B, Cin, Cout, H, W,
               _p(out), _stream())
    return out


def convT3x3_planes(planes, w_hi, w_lo, Cout, scale_bo=None):
    """conv_transpose2d(stride 2, pad 0) over key planes -> [B,Cout,2H+1,2W+1] fp32."""
    B, Cin, H, W = planes.B, planes.C, planes.H, planes.W
    out = torch.empty((B, Cout, 2 * H + 1, 2 * W + 1), dtype=torch.float32,
                      device=planes.hi.device)
    _cabi.call('rw_modconv_up_fwd', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo),
               _p(scale_bo), B, Cin, Cout, H, W, _p(out), _stream())
    return out


def blur_up_act(t, kernel, noise=None, noise_w=None, bias=None, act=False):
    t = _f32c(t)
    B, C, Ht, Wt = t.shape
    Hin, Win = (Ht - 1) // 2, (Wt - 1) // 2
    y = torch.empty((B, C, 2 * Hin, 2 * Win), dtype=torch.float32, device=t.device)
    nstride = noise.stride(0) if noise is not None else 0
    _cabi.call('rw_blur_up_act', _p(t), B, C, Hin, Win, _p(_f32c(kernel)), _p(noise), nstride,
               _p(noise_w), _p(bias), 1 if act else 0, _p(y), _stream())
    return y


def add_noise(x, noise, noise_w):
    x = _f32c(x)
    B, C, H, W = x.shape
    y = torch.empty_like(x)
    _cabi.call('rw_add_noise', _p(x), _p(noise), noise.stride(0), _p(_f32c(noise_w.detach())), B, C,
               H * W, _p(y), _stream())
    return y


def torgb(x, style, weight, bias, skip=None):
    """out = conv1x1(style*x, W/sqrt(C)) + bias (+ skip)   (ToRGBF, models.py:639-655)."""
    x = _f32c(x)
    B, C, H, W = x.shape
    out = torch.empty((B, 3, H, W), dtype=torch.float32, device=x.device)
    _cabi.call('rw_torgb', _p(x), _p(_f32c(style)), _p(_f32c(weight.reshape(3, C))),
               _p(_f32c(bias.reshape(3))), _p(_f32c(skip)), B, C, H, W, 1.0 / math.sqrt(C),
               _p(out), _stream())
    return out


def fused_bias_act_raw(x, bias, ref, act, grad, alpha, scale):
    """The reference's `fused.fused_bias_act` (op/fused_bias_act.cpp:11-21)."""
    x = _f32c(x)
    y = torch.empty_like(x)
    has_b = bias is not None and bias.numel() > 0
    has_r = ref is not None and ref.numel() > 0
    step_b = 1
    for i in range(2, x.dim()):
        step_b *= x.shape[i]
    _cabi.call('rw_fused_bias_act', _p(x), _p(_f32c(bias)) if has_b else None,
               _p(_f32c(ref)) if has_r else None, int(act), int(grad), float(alpha), float(scale),
               x.numel(), step_b, bias.numel() if has_b else 1, _p(y), _stream())
    return y


def upfirdn2d_raw(inp, kernel, up_x, up_y, down_x, down_y, px0, px1, py0, py1):
    """The reference's `upfirdn2d_op.upfirdn2d` on a [major, H, W, 1] view
    (op/upfirdn2d.cpp:4-22)."""
    inp = _f32c(inp)
    major, in_h, in_w, minor = inp.shape
    if minor != 1:
        inp = inp.permute(0, 3, 1, 2).contiguous()
        major_eff = major * minor
    else:
        major_eff = major
    kh, kw = kernel.shape
    out_h = (in_h * up_y + py0 + py1 - kh) // down_y + 1
    out_w = (in_w * up_x + px0 + px1 - kw) // down_x + 1
    out = torch.empty((major_eff, out_h, out_w), dtype=torch.float32, device=inp.device)
    _cabi.call('rw_upfirdn2d', _p(inp), _p(_f32c(kernel)), major_eff, in_h, in_w, kh, kw, up_x,
               up_y, down_x, down_y, px0, px1, py0, py1, _p(out), out_h, out_w, _stream())
    if minor != 1:
        return out.view(major, minor, out_h, out_w).permute(0, 2, 3, 1).contiguous()
    return out.view(major, out_h, out_w, 1)


# --------------------------------------------------------------------------- second moment
_WS = {}


def _workspace(nbytes, device):
    key = str(device)
    ws = _WS.get(key)
    if ws is None or ws.numel() * 4 < nbytes:
        ws = torch.empty((nbytes + 3) // 4 + 64, dtype=torch.float32, device=device)
        _WS[key] = ws
    return ws


def second_moment_accum_planes(mom2, hi, lo):
    """mom2 += hi/lo planes^T @ planes  (RunningSecondMoment.add, runningstats.py:1086-1097)."""
    rows, C = hi.shape
    lib = _cabi.load()
    ws = _workspace(lib.rw_gram_workspace_bytes(C, C, rows, 1), hi.device)
    _cabi.call('rw_second_moment_accum', _p(hi), _p(lo), rows, C, _p(mom2), _p(ws),
               ws.numel() * 4, _stream())


def second_moment_accum(mom2, a):
    hi, lo = split_rows(a)
    second_moment_accum_planes(mom2, hi, lo)


def conv_wgrad_planes(g_planes, k_planes):
    """dWt[o][tap][i] = sum_p G[p,o] K[p+shift(tap), i]  -> [Cout, 9, Cin] fp32."""
    rows = g_planes.rows
    Cout, Cin = g_planes.C, k_planes.C
    lib = _cabi.load()
    ws = _workspace(lib.rw_gram_workspace_bytes(Cout, Cin, rows, 9), g_planes.hi.device)
    out = torch.empty((Cout, 9, Cin), dtype=torch.float32, device=g_planes.hi.device)
    _cabi.call('rw_conv_wgrad', _p(g_planes.hi), _p(g_planes.lo), _p(k_planes.hi),
               _p(k_planes.lo), rows, Cout, Cin, k_planes.W + 1, _p(out), _p(ws), ws.numel() * 4,
               _stream())
    return out


# --------------------------------------------------------------------------- rank projection
def project_rank(weight, direction, base=None, sign=1.0):
    """base + sign * projected_conv(weight, direction)   (ganrewrite.py:806-813)."""
    w = _f32c(weight)
    d = _f32c(direction)
    shp = w.shape
    if w.dim() == 5:
        Cout, Cin, taps = shp[1], shp[2], shp[3] * shp[4]
        assert shp[0] == 1
    else:
        Cout, Cin, taps = shp[0], shp[1], shp[2] * shp[3]
    rank = d.shape[0]
    out = torch.empty_like(w)
    _cabi.call('rw_project_rank', _p(w), _p(_f32c(base)), _p(d), rank, Cout, Cin, taps,
               float(sign), _p(out), _stream())
    return out


# --------------------------------------------------------------------------- autograd
LRELU_SLOPE = 0.2
LRELU_GAIN = 2 ** 0.5


class StyledConvFunction(torch.autograd.Function):
    """y = [act]([blur](conv(style*x, scale*W) * demod) + nw*noise + bias)

    One fused forward (prep -> tcgen05 row-GEMM with fused epilogue); backward =
    dgrad row-GEMM on gradient planes + wgrad col-GEMM + small reductions.
    """

    @staticmethod
    def forward(ctx, x, style, weight, noise_weight, bias, upsample, blur_kernel, demodulate,
                with_noise, with_act, pre_modulated, wholder):
        x = _f32c(x)
        style = _f32c(style)
        B, Cin, H, W = x.shape
        Cout = weight.shape[-4]
        if pre_modulated:
            planes, _ = prep_keys(x, None)
        else:
            planes, _ = prep_keys(x, style)
        w_hi, w_lo, wsq = wholder.planes('fwd')
        dm = demod_factors(style, wsq) if demodulate else None
        # device scalar: the kernels read the Parameter's storage (no .item() host sync)
        nw = _f32c(noise_weight.detach()) if (with_noise and noise_weight is not None) else None
        if nw is None:
            with_noise = False
        b = _f32c(bias.detach()) if (with_act and bias is not None) else None
        if upsample and up_fused_eligible(Cin, Cout, H, W, blur_kernel):
            # the whole layer in one launch (csrc/upconv_tc.cu, layer-level mode: y as fp32 NCHW);
            # backward only needs y (the leaky-ReLU gate) and the planes
            noise = noise_table(B, 4 * H * W, x.device) if with_noise else None
            u_hi, u_lo, _ = wholder.planes('upf')
            y = torch.empty((B, Cout, 2 * H, 2 * W), dtype=torch.float32, device=x.device)
            kern = _f32c(blur_kernel)
            _cabi.call('rw_modconv_up_fused_y', _p(planes.hi), _p(planes.lo), _p(u_hi), _p(u_lo),
                       _p(dm) if dm is not None else None, _p(kern),
                       _p(noise) if with_noise else None, noise.stride(0) if with_noise else 0,
                       _p(nw) if with_noise else None, _p(b) if b is not None else None,
                       1 if with_act else 0, _p(y), B, Cin, Cout, H, W, _stream())
        elif upsample:
            t_up = convT3x3_planes(planes, w_hi, w_lo, Cout, dm)
            Ho, Wo = 2 * H, 2 * W
            noise = noise_table(B, Ho * Wo, x.device) if with_noise else None
            y = blur_up_act(t_up, blur_kernel, noise, nw, b, with_act)
        else:
            noise = noise_table(B, H * W, x.device) if with_noise else None
            y = conv3x3_planes(planes, w_hi, w_lo, Cout, dm, noise, nw, b, with_act)
        ctx.save_for_backward(x, style, weight, noise_weight, bias, y, dm)
        ctx.cfg = (upsample, demodulate, with_noise, with_act, pre_modulated)
        ctx.blur_kernel = blur_kernel
        ctx.wholder = wholder
        ctx.planes = planes if any(ctx.needs_input_grad) else None
        return y

    @staticmethod
    def backward(ctx, gy):
        """Five HBM passes + two tensor-core GEMMs (csrc/bwd.cu):
        act_grad_reduce (gy, y -> g_pre and every per-(b,o) reduction) -> gradient planes
        (prep_keys, or blur^T + phase split for up layers) -> dgrad row-GEMM -> dgrad_finish
        (gx, dstyle) ; wgrad col-GEMM -> wgrad_finish (demodulation term, Parameter layout)."""
        x, style, weight, noise_weight, bias, y, dm = ctx.saved_tensors
        upsample, demodulate, with_noise, with_act, pre_modulated = ctx.cfg
        if ctx.planes is None:
            raise _cabi.RwError('StyledConvFunction.backward: forward ran without autograd state')
        need_x, need_style, need_w = ctx.needs_input_grad[:3]
        gy = _f32c(gy)
        B, Cin, H, W = x.shape
        Cout = weight.shape[-4]
        sc = 1.0 / math.sqrt(Cin * 9)
        Ho, Wo = (2 * H, 2 * W) if upsample else (H, W)
        dev = x.device
        has_noise = with_noise and noise_weight is not None
        has_bias = with_act and bias is not None
        noise = noise_table(B, Ho * Wo, dev) if has_noise else None
        nw = _f32c(noise_weight.detach()) if has_noise else None
        bv = _f32c(bias.detach()) if has_bias else None
        # one pass over (gy, y): gradient through the activation (gate on the sign of the saved
        # output) and the three per-(b,o) pixel reductions
        red = torch.empty((3, B, Cout), dtype=torch.float32, device=dev)
        g_pre = torch.empty_like(gy) if with_act else None
        _cabi.call('rw_act_grad_reduce', _p(gy), _p(y), _p(noise),
                   noise.stride(0) if has_noise else 0, _p(nw), _p(bv), 1 if with_act else 0,
                   B, Cout, Ho * Wo, _p(g_pre), _p(red[0]), _p(red[1]), _p(red[2]), _stream())
        if g_pre is None:
            g_pre = gy
        g_bias = red[0].sum(dim=0) if has_bias else None
        g_nw = red[2].sum().reshape(noise_weight.shape) if has_noise else None
        s_dot = red[1] if demodulate else None        # = dL/d(demod) * demod
        k_planes = ctx.planes
        need_dk = need_x or (need_style and not pre_modulated)
        dk = dwt = None
        if upsample:
            rows = B * (H + 1) * (W + 1)
            gph_hi = torch.empty((rows, 4 * Cout), dtype=torch.bfloat16, device=dev)
            gph_lo = torch.empty_like(gph_hi)
            # blur^T(g_pre) * demod, split into the 4 conv_transpose phases
            _cabi.call('rw_blur_adj_phase_keys', _p(g_pre), _p(dm), _p(_f32c(ctx.blur_kernel)), B,
                       Cout, H, W, _p(gph_hi), _p(gph_lo), _stream())
            if need_dk:
                wd_hi, wd_lo, _ = ctx.wholder.planes('dgrad_up')
                dk = torch.empty((B, Cin, H, W), dtype=torch.float32, device=dev)
                _cabi.call('rw_modconv_up_dgrad', _p(gph_hi), _p(gph_lo), _p(wd_hi), _p(wd_lo),
                           None, B, Cin, Cout, H, W, _p(dk), _stream())
            if need_w:
                lib = _cabi.load()
                ws = _workspace(lib.rw_gram_workspace_bytes(Cout, Cin, rows, 9), dev)
                dwt = torch.empty((Cout, 9, Cin), dtype=torch.float32, device=dev)
                _cabi.call('rw_conv_up_wgrad', _p(gph_hi), _p(gph_lo), _p(k_planes.hi),
                           _p(k_planes.lo), rows, Cout, Cin, W + 1, _p(dwt), _p(ws),
                           ws.numel() * 4, _stream())
        else:
            g_planes, _ = prep_keys(g_pre, dm)          # planes of g_t = g_pre * demod
            if need_dk:
                wd_hi, wd_lo, _ = ctx.wholder.planes('dgrad')
                dk = conv3x3_planes(g_planes, wd_hi, wd_lo, Cin)   # conv(g_t, flip(W)^T)
            if need_w:
                dwt = conv_wgrad_planes(g_planes, k_planes)        # [Cout, 9, Cin]
        gx = g_style = gs_raw = None
        if need_dk:
            if pre_modulated:
                gx = dk
            else:
                gs_raw = torch.empty((B, Cin), dtype=torch.float32, device=dev)
                _cabi.call('rw_dgrad_finish', _p(dk), _p(x), _p(style), B, Cin, H * W, _p(gs_raw),
                           _stream())
                gx = dk                                  # scaled by style in place
        if need_style and (gs_raw is not None or demodulate):
            wsq = ctx.wholder.planes('fwd')[2] if demodulate else None
            g_style = torch.empty((B, Cin), dtype=torch.float32, device=dev)
            _cabi.call('rw_style_grad_finish', _p(gs_raw), _p(style), _p(s_dot), _p(dm), _p(wsq),
                       B, Cout, Cin, _p(g_style), _stream())
        gW = None
        if need_w:
            gW = torch.empty(weight.shape, dtype=torch.float32, device=dev)
            _cabi.call('rw_wgrad_finish', _p(dwt), _p(_f32c(weight.detach())), _p(s_dot), _p(dm),
                       _p(style), B, Cout, Cin, sc, _p(gW), _stream())
        return gx, g_style, gW, g_nw, g_bias, None, None, None, None, None, None, None


class _WeightHolder(object):
    """Carries the caller's weight OBJECT into the autograd Function so that the plane cache
    is keyed on the user's Parameter, not on whatever view autograd hands to forward()."""
    __slots__ = ('weight',)

    def __init__(self, weight):
        self.weight = weight

    def planes(self, kind):
        return weight_planes(self.weight, kind)


class ConvTransposeLeafFunction(torch.autograd.Function):
    """t = conv_transpose2d(k, scale*W^T, stride 2) * demod(W, style) on an already-modulated key
    — the `dconv` LEAF of an upsampling layer when nethook has split the layer at it (the blur
    is then the next leaf): reference DemodulatedConv2dF.forward, models.py:313-329, upsample
    branch.  Differentiable in the weight (incl. the demodulation term) and in the key, which is
    what the rewriter's edit of an odd layer needs (ganrewrite.py:254-298); the style enters only
    through demod and gets no gradient here (the rewriter detaches it)."""

    @staticmethod
    def forward(ctx, k, style, weight, demodulate, wholder):
        k = _f32c(k)
        style = _f32c(style)
        B, Cin, H, W = k.shape
        Cout = weight.shape[-4]
        planes, _ = prep_keys(k, None)
        w_hi, w_lo, wsq = wholder.planes('fwd')
        dm = demod_factors(style, wsq) if demodulate else None
        out = convT3x3_planes(planes, w_hi, w_lo, Cout, dm)
        ctx.save_for_backward(style, weight, out, dm)
        ctx.planes = planes if any(ctx.needs_input_grad) else None
        ctx.wholder = wholder
        ctx.shape = (B, Cin, Cout, H, W)
        return out

    @staticmethod
    def backward(ctx, gt):
        style, weight, out, dm = ctx.saved_tensors
        B, Cin, Cout, H, W = ctx.shape
        need_k, _, need_w = ctx.needs_input_grad[:3]
        gt = _f32c(gt)
        dev = gt.device
        rows = B * (H + 1) * (W + 1)
        gph_hi = torch.empty((rows, 4 * Cout), dtype=torch.bfloat16, device=dev)
        gph_lo = torch.empty_like(gph_hi)
        # phase planes of g_t * demod over the input-resolution padded grid
        _cabi.call('rw_prep_phase_keys', _p(gt), _p(dm), B, Cout, H, W, _p(gph_hi), _p(gph_lo),
                   _stream())
        gk = gW = None
        if need_k:
            wd_hi, wd_lo, _ = ctx.wholder.planes('dgrad_up')
            gk = torch.empty((B, Cin, H, W), dtype=torch.float32, device=dev)
            _cabi.call('rw_modconv_up_dgrad', _p(gph_hi), _p(gph_lo), _p(wd_hi), _p(wd_lo), None, B,
                       Cin, Cout, H, W, _p(gk), _stream())
        if need_w:
            lib = _cabi.load()
            ws = _workspace(lib.rw_gram_workspace_bytes(Cout, Cin, rows, 9), dev)
            dwt = torch.empty((Cout, 9, Cin), dtype=torch.float32, device=dev)
            _cabi.call('rw_conv_up_wgrad', _p(gph_hi), _p(gph_lo), _p(ctx.planes.hi),
                       _p(ctx.planes.lo), rows, Cout, Cin, W + 1, _p(dwt), _p(ws), ws.numel() * 4,
                       _stream())
            # dL/d(demod) * demod = sum_pixels g_t * t  (t is the saved, demodulated output)
            s_dot = (gt * out).sum(dim=(2, 3)).contiguous() if dm is not None else None
            gW = torch.empty(weight.shape, dtype=torch.float32, device=dev)
            _cabi.call('rw_wgrad_finish', _p(dwt), _p(_f32c(weight.detach())), _p(s_dot), _p(dm),
                       _p(style), B, Cout, Cin, 1.0 / math.sqrt(Cin * 9), _p(gW), _stream())
        return gk, None, gW, None, None


def conv_transpose_leaf(k, style, weight, demodulate=True):
    return ConvTransposeLeafFunction.apply(k, style, weight, demodulate, _WeightHolder(weight))


def styled_conv(x, style, weight, noise_weight=None, bias=None, upsample=False, blur_kernel=None,
                demodulate=True, with_noise=True, with_act=True, pre_modulated=False):
    return StyledConvFunction.apply(x, style, weight, noise_weight, bias, upsample, blur_kernel,
                                    demodulate, with_noise, with_act, pre_modulated,
                                    _WeightHolder(weight))


# --------------------------------------------------------------------------- ProgGAN leaves
def pixel_norm_nchw(x, up2=False):
    """PixelNormLayer (reference utils/proggan.py:128-134), optionally fused with the nearest 2x
    of the DoubleResolutionLayer that follows it in NormUpscaleConvBlock (:137-141)."""
    x = _f32c(x)
    B, C, H, W = x.shape
    out = torch.empty((B, C, 2 * H, 2 * W) if up2 else (B, C, H, W), dtype=torch.float32,
                      device=x.device)
    _cabi.call('rw_pixel_norm_nchw', _p(x), B, C, H, W, 1 if up2 else 0, _p(out), _stream())
    return out


def nearest_up2(x):
    x = _f32c(x)
    B, C, H, W = x.shape
    out = torch.empty((B, C, 2 * H, 2 * W), dtype=torch.float32, device=x.device)
    _cabi.call('rw_nearest_up2', _p(x), B * C, H, W, _p(out), _stream())
    return out


def plain_conv_eligible(weight):
    return (weight.dim() == 4 and weight.shape[2] == 3 and weight.shape[3] == 3 and
            weight.shape[0] % 128 == 0 and weight.shape[1] % 64 == 0)


def conv3x3_bias_act(x, weight, wscale=1.0, bias=None, act=False, act_gain=1.0):
    """lrelu(conv3x3(x, wscale * W) + bias) on the tensor-core row-GEMM, no autograd: the fused
    NormConvBlock tail conv -> WScaleLayer -> LeakyReLU (proggan.py:158-181)."""
    planes, _ = prep_keys(x, None)
    w_hi, w_lo, _ = weight_planes(weight, 'fwd', scale=wscale)
    B, Cin, H, W = planes.B, planes.C, planes.H, planes.W
    Cout = weight.shape[0]
    out = torch.empty((B, Cout, H, W), dtype=torch.float32, device=planes.hi.device)
    _cabi.call('rw_conv3x3_bias_act', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo),
               _p(_f32c(bias.detach()) if bias is not None else None), 1 if act else 0,
               float(act_gain), B, Cin, Cout, H, W, _p(out), _stream())
    return out


class PlainConvFunction(torch.autograd.Function):
    """y = conv3x3(x, W) (pad 1, no bias) — the `layerN.conv` target of ProgressiveGanRewriter —
    forward and backward on the same tensor-core kernels as the styled conv (row-GEMM for y and
    dX, col-GEMM for dW), weight scale 1."""

    @staticmethod
    def forward(ctx, x, weight, wholder):
        x = _f32c(x)
        planes, _ = prep_keys(x, None)
        w_hi, w_lo, _ = weight_planes(wholder.weight, 'fwd', scale=1.0)
        y = conv3x3_planes(planes, w_hi, w_lo, weight.shape[0])
        ctx.save_for_backward(weight)
        ctx.planes = planes if any(ctx.needs_input_grad) else None
        ctx.wholder = wholder
        return y

    @staticmethod
    def backward(ctx, gy):
        (weight,) = ctx.saved_tensors
        need_x, need_w = ctx.needs_input_grad[:2]
        g_planes, _ = prep_keys(_f32c(gy), None)
        Cout, Cin = weight.shape[0], weight.shape[1]
        gx = gW = None
        if need_x:
            wd_hi, wd_lo, _ = weight_planes(ctx.wholder.weight, 'dgrad', scale=1.0)
            gx = conv3x3_planes(g_planes, wd_hi, wd_lo, Cin)
        if need_w:
            dwt = conv_wgrad_planes(g_planes, ctx.planes)            # [Cout, 9, Cin]
            gW = torch.empty(weight.shape, dtype=torch.float32, device=gy.device)
            _cabi.call('rw_wgrad_finish', _p(dwt), _p(_f32c(weight.detach())), None, None, None,
                       g_planes.B, Cout, Cin, 1.0, _p(gW), _stream())
        return gx, gW, None


def plain_conv(x, weight):
    return PlainConvFunction.apply(x, weight, _WeightHolder(weight))


# --------------------------------------------------------------------------- key algebra
def rowgemm(a, w_planes):
    """a [M, K] fp32 (CUDA) times W^T for W [N, K] given as (hi, lo) planes from split_rows:
    out [M, N] on the tensor-core row-GEMM (no cuBLAS between key capture and d)."""
    a = _f32c(a)
    M, K = a.shape
    w_hi, w_lo = w_planes
    N = w_hi.shape[0]
    a_hi, a_lo = split_rows(a)
    out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    _cabi.call('rw_rowgemm', _p(a_hi), _p(a_lo), _p(w_hi), _p(w_lo), M, K, N, _p(out), _stream())
    return out
