"""Generation fast path of an intact SeqStyleGAN2: producers write the consumer's operands.

The layer-by-layer execution (`StyledConvSeq.forward`) has to hand an fp32 NCHW feature map to
whatever comes next (a hook, a nethook slice, ToRGB, the next layer's prep), which costs three
extra passes over every activation.  When the WHOLE generator runs unhooked and without
autograd, nothing observes those tensors, so this module chains the kernels directly:

    planes(L) --conv_tc--> epilogue { lrelu(..)·√2 ; x next style -> planes(L+1) ; ToRGB partial }
    planes(L) --conv_tc(4 phases)--> t (channels-last) --blur_up_fused--> planes(L+1)
    rgb partials --rgb_combine--> running image (+ bias + 2x-upsampled skip)

The arithmetic per element is the same as the layer path (same kernels, same fp32 epilogue
expressions), only the intermediate fp32 tensors are never materialised.  Also serves the
rewriter's key collection: `upto_key_layer=N` stops in front of `layerN`'s convolution and returns
its key planes, which are exactly the operands of the second-moment GEMM.

Reference semantics: SeqStyleGAN2.forward, utils/stylegan2/models.py:92-141.
"""
import ctypes
import math

import torch

from . import _cabi, ops
from .ops import _p, _stream


def _layer_list(model):
    """[(layer number, StyledConvSeq, latent index, ToRGBF or None, rgb latent index)] in order,
    or None if the module tree is not the pristine SeqStyleGAN2 layout."""
    from .utils.stylegan2 import models as sg2
    names = list(model._modules.keys())
    expect = ['bag_in', 'style', 'latents', 'noises', 'input', 'layer2', 'to_rgb1']
    n = 3
    for k in range(1, model.log_size - 1):
        expect += ['up_rgb%d' % k, 'layer%d' % n, 'layer%d' % (n + 1), 'to_rgb%d' % (k + 1)]
        n += 2
    expect.append('output')
    if names != expect:
        return None
    out = []
    for name in names:
        if not name.startswith('layer'):
            continue
        num = int(name[5:])
        seq = model._modules[name]
        kids = list(seq._modules.items())
        if len(kids) != 2 or not isinstance(kids[0][1], sg2.PickLatent):
            return None
        sconv = kids[1][1]
        if not isinstance(sconv, sg2.StyledConvSeq):
            return None
        mc = sconv._modules.get('mconv')
        if not isinstance(mc, sg2.ModulatedConv2dSeq):
            return None
        want = ['modulation', 'adain', 'dconv'] + (['blur'] if mc.upsample else [])
        if list(mc._modules.keys()) != want or list(sconv._modules.keys()) != ['mconv', 'noise', 'activate']:
            return None
        if mc.dconv.kernel_size != 3 or not mc.dconv.demodulate:
            return None
        rgb = None
        rgb_lat = None
        if num % 2 == 0:
            rseq = model._modules['to_rgb%d' % (num // 2)]
            rk = list(rseq._modules.items())
            if len(rk) != 2 or not isinstance(rk[1][1], sg2.ToRGBF):
                return None
            rgb, rgb_lat = rk[1][1], rk[0][1].index
        out.append((num, sconv, kids[0][1].index, rgb, rgb_lat))
    return out


def eligible(model, z):
    from .utils.stylegan2 import models as sg2
    if not isinstance(z, torch.Tensor) or z.dim() != 2 or not z.is_cuda or z.dtype != torch.float32:
        return False
    if model.bag_input or model.bag_output or model.mconv != 'seq':
        return False
    if torch.is_grad_enabled() and (z.requires_grad or any(p.requires_grad for p in model.parameters())):
        return False
    if sg2._is_hooked(model):
        return False
    return _layer_list(model) is not None


import os as _os

# RW_UP_FUSED=0 keeps the round-1 pair (conv_transpose phases -> channels-last t -> blur kernel);
# RW_UP_FUSED_MINW = smallest input width that takes the fused kernel
_UP_FUSED = _os.environ.get('RW_UP_FUSED', '1') != '0'
_UP_FUSED_MINW = int(_os.environ.get('RW_UP_FUSED_MINW', '4'))


def _use_fused_up(mc, Cin, Cout, H, W):
    return (_UP_FUSED and H == W and _UP_FUSED_MINW <= W <= 128 and (W & (W - 1)) == 0 and
            Cin % 64 == 0 and Cout % 16 == 0 and ops.blur_is_separable(mc.blur.kernel))


def _mapping(model, z, stream):
    """w = AdjustLatent(style MLP(z)) as [B, style_dim] (models.py:487-533,570-583,609-614):
    PixelNorm + one fused EqualLinear(lrelu) launch per layer instead of sgemm + bias_act + two
    elementwise kernels each.  All n_latent copies of the reference's `latent` are this row."""
    from .utils.stylegan2 import models as sg2
    mods = list(model.style._modules.values())
    pristine = (len(mods) > 1 and isinstance(mods[0], sg2.PixelNormL) and
                all(type(m) is sg2.EqualLinearL and m.activation and m.bias is not None
                    for m in mods[1:]))
    if not pristine:
        return model.latents(model.style(model.bag_in(z))).latent[:, 0].contiguous()
    z = z.contiguous()
    B, K = z.shape
    x = torch.empty_like(z)
    _cabi.call('rw_pixel_norm', _p(z), B, K, _p(x), stream)
    for m in mods[1:]:
        cout, kin = m.weight.shape
        out = torch.empty((B, cout), dtype=torch.float32, device=z.device)
        _cabi.call('rw_equal_linear', _p(x), B, kin, _p(m.weight), _p(m.bias), cout,
                   float(m.scale), float(m.lr_mul), 1, _p(out), stream)
        x = out
    lat = model.latents
    if lat.truncation != 1.0 and lat.latent_avg.ndim > 0:      # AdjustLatent.forward
        x = lat.latent_avg + lat.truncation * (x - lat.latent_avg)
    return x


def forward(model, z, upto_key_layer=None, noise_period=None, out_u8=False):
    """image [B,3,size,size] (or KeyPlanes of `layer<upto_key_layer>`'s key).
    `noise_period`: sample i takes the noise row (i % noise_period) — see ops.noise_table.
    `out_u8`: return the image as NHWC uint8, clamp(x*127.5+127.5, 0, 255), written by the last
    ToRGB combine (the fp32 image is then never stored)."""
    from .utils import nvtx
    with nvtx.range('rw:generator' if upto_key_layer is None else 'rw:context'):
        return _forward(model, z, upto_key_layer, noise_period, out_u8)


def _forward(model, z, upto_key_layer, noise_period, out_u8):
    from .utils.stylegan2 import models as sg2
    layers = _layer_list(model)
    if layers is None:
        raise _cabi.RwError('fastpath: the module tree is not a pristine SeqStyleGAN2')
    dev = z.device
    B = z.shape[0]
    stream = _stream()
    w_lat = _mapping(model, z, stream)                   # [B, 512]: every latent slot is this row
    K = w_lat.shape[1]
    run = [l for l in layers if upto_key_layer is None or l[0] < upto_key_layer]
    if upto_key_layer is not None:
        # key collection: the running RGB image feeds nothing, skip every ToRGB; layers past the
        # key layer are never run, so neither their styles nor their demodulation factors are
        # computed (the key layer's own style scales the last producer's output planes)
        layers = [(num, sconv, lat, None, None) for num, sconv, lat, _, _ in layers
                  if num <= upto_key_layer]
        run = [(num, sconv, lat, None, None) for num, sconv, lat, _, _ in run]
        if not layers or layers[-1][0] != upto_key_layer:
            raise ValueError('layer%s not found' % upto_key_layer)

    # all styles up front (they only depend on the latent): ONE launch for the 13 + 7
    # modulation linears instead of 20 tiny sgemms
    mods = []
    for num, sconv, lat, rgb, rgb_lat in layers:
        mods.append((('conv', num), sconv.mconv.modulation, lat))
        if rgb is not None:
            mods.append((('rgb', num), rgb.conv.modulation, rgb_lat))
    n = len(mods)
    outs = [torch.empty((B, m.weight.shape[0]), dtype=torch.float32, device=dev) for _, m, _ in mods]
    PtrArr, IntArr = ctypes.c_void_p * n, ctypes.c_int * n
    _cabi.call('rw_styles', _p(w_lat), B, 1, K, float(mods[0][1].scale), n,
               PtrArr(*[m.weight.data_ptr() for _, m, _ in mods]),
               PtrArr(*[m.bias.data_ptr() for _, m, _ in mods]),
               PtrArr(*[o.data_ptr() for o in outs]),
               IntArr(*([0] * n)),
               IntArr(*[m.weight.shape[0] for _, m, _ in mods]), stream)
    styles, rgb_styles = {}, {}
    for (kind, num), o in zip([k for k, _, _ in mods], outs):
        (styles if kind == 'conv' else rgb_styles)[num] = o

    # ... and everything else that only depends on the styles: the demodulation factors of every
    # conv and ToRGB's modulated 1x1 weights, one launch
    demods, rgb_ws, jobs = {}, {}, []
    for num, sconv, lat, rgb, rgb_lat in run:
        dconv = sconv.mconv.dconv
        wsq = ops.weight_planes(dconv.weight, 'fwd')[2]
        demods[num] = torch.empty((B, dconv.out_channel), dtype=torch.float32, device=dev)
        jobs.append((styles[num], wsq, demods[num], dconv.out_channel, dconv.in_channel, 0, 1.0))
        if rgb is not None:
            C = dconv.out_channel
            rgb_ws[num] = torch.empty((B, 3, C), dtype=torch.float32, device=dev)
            jobs.append((rgb_styles[num], rgb.conv.weight.detach().reshape(3, C), rgb_ws[num], 3, C,
                         1, 1.0 / math.sqrt(C)))
    if jobs:
        nj = len(jobs)
        P, I, Fl = ctypes.c_void_p * nj, ctypes.c_int * nj, ctypes.c_float * nj
        _cabi.call('rw_demod_multi', B, 1e-8, nj, P(*[j[0].data_ptr() for j in jobs]),
                   P(*[j[1].data_ptr() for j in jobs]), P(*[j[2].data_ptr() for j in jobs]),
                   I(*[j[3] for j in jobs]), I(*[j[4] for j in jobs]), I(*[j[5] for j in jobs]),
                   Fl(*[j[6] for j in jobs]), stream)

    x0 = model.input.input
    H = W = x0.shape[2]
    first = layers[0]
    planes, _ = ops.prep_keys(x0.repeat(B, 1, 1, 1), styles[first[0]])
    if upto_key_layer == first[0]:
        return planes
    image = None
    for idx, (num, sconv, lat, rgb, rgb_lat) in enumerate(layers):
        if upto_key_layer == num:
            return planes
        mc = sconv.mconv
        dconv = mc.dconv
        Cin, Cout = dconv.in_channel, dconv.out_channel
        w_hi, w_lo, _ = ops.weight_planes(dconv.weight, 'fwd')
        dm = demods[num]
        nxt = layers[idx + 1] if idx + 1 < len(layers) else None
        next_scale = styles[nxt[0]] if nxt is not None else None
        nw = sconv.noise.weight.detach()
        bias = sconv.activate.bias.detach()
        if mc.upsample and _use_fused_up(mc, Cin, Cout, H, W):
            # conv_transpose + blur + noise + bias + act + next style in ONE tensor-core kernel
            u_hi, u_lo, _ = ops.weight_planes(dconv.weight, 'upf')
            Ho, Wo = 2 * H, 2 * W
            noise = ops.noise_table(B, Ho * Wo, dev, noise_period)
            rows_o = B * (Ho + 1) * (Wo + 1)
            nh = torch.empty((rows_o, Cout), dtype=torch.bfloat16, device=dev)
            nl = torch.empty_like(nh)
            _cabi.call('rw_modconv_up_fused', _p(planes.hi), _p(planes.lo), _p(u_hi), _p(u_lo),
                       _p(dm), _p(mc.blur.kernel), _p(noise), noise.stride(0), _p(nw), _p(bias),
                       _p(next_scale), _p(nh), _p(nl), B, Cin, Cout, H, W, stream)
            H, W = Ho, Wo
            planes = ops.KeyPlanes(nh, nl, B, Cout, H, W)
        elif mc.upsample:
            rows = B * (H + 1) * (W + 1)
            t_cl = torch.empty((4, rows, Cout), dtype=torch.float32, device=dev)
            _cabi.call('rw_modconv_up_fwd_cl', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo),
                       _p(dm), B, Cin, Cout, H, W, _p(t_cl), stream)
            Ho, Wo = 2 * H, 2 * W
            noise = ops.noise_table(B, Ho * Wo, dev, noise_period)
            rows_o = B * (Ho + 1) * (Wo + 1)
            nh = torch.empty((rows_o, Cout), dtype=torch.bfloat16, device=dev)
            nl = torch.empty_like(nh)
            _cabi.call('rw_blur_up_fused', _p(t_cl), B, Cout, H, W, _p(mc.blur.kernel), _p(noise),
                       noise.stride(0), _p(nw), _p(bias), 1, _p(next_scale), _p(nh), _p(nl), None,
                       stream)
            H, W = Ho, Wo
            planes = ops.KeyPlanes(nh, nl, B, Cout, H, W)
        else:
            noise = ops.noise_table(B, H * W, dev, noise_period)
            rows = B * (H + 1) * (W + 1)
            nh = nl = None
            if nxt is not None:
                nh = torch.empty((rows, Cout), dtype=torch.bfloat16, device=dev)
                nl = torch.empty_like(nh)
            rgb_w = rgb_part = None
            ntile = 0
            if rgb is not None:
                ntile = ops.rgb_parts(Cout)     # one ToRGB partial per epilogue column group
                rgb_w = rgb_ws[num]                                              # [B,3,Cout]
                rgb_part = torch.empty((ntile, B, 3, H, W), dtype=torch.float32, device=dev)
            _cabi.call('rw_modconv_fwd_fused', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo),
                       _p(dm), _p(noise), noise.stride(0), _p(nw), _p(bias), 1, B, Cin, Cout, H, W,
                       None, _p(next_scale), _p(nh), _p(nl), _p(rgb_w), _p(rgb_part), stream)
            if rgb is not None:
                last = out_u8 and nxt is None
                out = None if last else torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
                up_k = None
                if image is not None:
                    up_k = model._modules['up_rgb%d' % (num // 2 - 1)].kernel
                if last:
                    out = torch.empty((B, H, W, 3), dtype=torch.uint8, device=dev)
                    _cabi.call('rw_rgb_combine_u8', _p(rgb_part), ntile, B, H, W,
                               _p(rgb.bias.detach().reshape(3).contiguous()), _p(image), _p(up_k),
                               None, _p(out), stream)
                else:
                    _cabi.call('rw_rgb_combine', _p(rgb_part), ntile, B, H, W,
                               _p(rgb.bias.detach().reshape(3).contiguous()), _p(image), _p(up_k),
                               _p(out), stream)
                image = out
            if nxt is not None:
                planes = ops.KeyPlanes(nh, nl, B, Cout, H, W)
    if upto_key_layer is not None:
        raise ValueError('layer%s not found' % upto_key_layer)
    return image
