"""Throughput of the 512^2 and 1024^2 StyleGAN2 generators (seeded weights) on one GPU.

    python tools/bench_highres.py [--steps 10] [--warmup 3] [--out profiles/r3_highres_b200.json]

Prints one JSON line:
  * img/s of the 1024^2 generator at batch 8 and 16 and of the 512^2 generator at batch 16,
    inputs resident (fp32 images stay on the device) and end to end (uint8 NHWC copied to pinned
    host memory); the L2 is overwritten between timed steps (as bench.py does);
  * per-layer kernel time of layers 13-18 of the 1024^2 generator at batch 8 (CUDA events around
    the same C-ABI launches the fast path makes), with the FLOP and HBM bytes computed from the
    shapes, the achieved rates and which of the two bounds the layer (B200 data sheet: 2.25
    PFLOP/s dense BF16, 7.7 TB/s);
  * the CPU oracle's s/img at 512^2;
  * the card name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_FLOPS = 2.25e15
PEAK_BYTES = 7.7e12


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                      # noqa: BLE001
        return 'unavailable: %s' % e


def seeded(size):
    from oracle import sg2_oracle as orc
    from rewriting_b200.utils.stylegan2 import SeqStyleGAN2
    return orc.seeded_state_dict(lambda: SeqStyleGAN2(size, style_dim=512, n_mlp=8, mconv='seq')).eval()


def gen_rate(model, B, steps, warmup, flush):
    from rewriting_b200 import fastpath
    from rewriting_b200.utils import zdataset
    z = zdataset.standard_z_sample(B, 512, seed=3).cuda()
    host = torch.empty((B, model.size, model.size, 3), dtype=torch.uint8).pin_memory()
    with torch.no_grad():
        for _ in range(warmup):
            fastpath.forward(model, z)
            host.copy_(fastpath.forward(model, z, out_u8=True))
        torch.cuda.synchronize()
        t_res = 0.0
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fastpath.forward(model, z)
            b.record()
            torch.cuda.synchronize()
            t_res += a.elapsed_time(b) / 1e3
        t_e2e = 0.0
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host.copy_(fastpath.forward(model, z, out_u8=True))
            torch.cuda.synchronize()
            t_e2e += time.perf_counter() - t0
    return B * steps / t_res, B * steps / t_e2e


def layer_launches(model, num, B):
    """(closure making the fast path's launches of layer `num`, FLOP, minimum HBM bytes)."""
    from rewriting_b200 import _cabi, fastpath, ops
    from rewriting_b200.ops import _p, _stream
    layers = {l[0]: l for l in fastpath._layer_list(model)}
    _, sconv, _, rgb, _ = layers[num]
    mc = sconv.mconv
    dconv = mc.dconv
    Cin, Cout = dconv.in_channel, dconv.out_channel
    res_out = 4 * 2 ** ((num - 1) // 2)            # layer 2: 4^2; layers 2k-1, 2k: 4 * 2^(k-1)
    H = W = res_out // 2 if mc.upsample else res_out
    dev = 'cuda'
    x = torch.randn(B, Cin, H, W, device=dev)
    style = torch.rand(B, Cin, device=dev) + 0.5
    planes = ops.prep_keys(x, style)[0]
    w_hi, w_lo, wsq = ops.weight_planes(dconv.weight, 'fwd')
    dm = ops.demod_factors(style, wsq)
    nw = sconv.noise.weight.detach()
    bias = sconv.activate.bias.detach()
    nscale = torch.rand(B, Cout, device=dev) + 0.5
    flop = 2.0 * B * H * W * Cin * Cout * 9
    if mc.upsample:
        Ho, Wo = 2 * H, 2 * W
        noise = ops.noise_table(B, Ho * Wo, dev)
        rows_o = B * (Ho + 1) * (Wo + 1)
        nh = torch.empty((rows_o, Cout), dtype=torch.bfloat16, device=dev)
        nl = torch.empty_like(nh)
        kern = mc.blur.kernel
        if fastpath._use_fused_up(mc, Cin, Cout, H, W):
            u_hi, u_lo, _ = ops.weight_planes(dconv.weight, 'upf')

            def run():
                _cabi.call('rw_modconv_up_fused', _p(planes.hi), _p(planes.lo), _p(u_hi), _p(u_lo),
                           _p(dm), _p(kern), _p(noise), noise.stride(0), _p(nw), _p(bias),
                           _p(nscale), _p(nh), _p(nl), B, Cin, Cout, H, W, _stream())
            nbytes = planes.rows * Cin * 4 + rows_o * Cout * 4
            return run, flop, nbytes, 'fused up'
        t_cl = torch.empty((4, planes.rows, Cout), dtype=torch.float32, device=dev)

        def run():
            _cabi.call('rw_modconv_up_fwd_cl', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo),
                       _p(dm), B, Cin, Cout, H, W, _p(t_cl), _stream())
            _cabi.call('rw_blur_up_fused', _p(t_cl), B, Cout, H, W, _p(kern), _p(noise),
                       noise.stride(0), _p(nw), _p(bias), 1, _p(nscale), _p(nh), _p(nl), None,
                       _stream())
        nbytes = planes.rows * Cin * 4 + 2 * t_cl.numel() * 4 + rows_o * Cout * 4
        return run, flop, nbytes, 'conv_transpose phases + blur'
    noise = ops.noise_table(B, H * W, dev)
    nh = torch.empty((planes.rows, Cout), dtype=torch.bfloat16, device=dev)
    nl = torch.empty_like(nh)
    nparts = ops.rgb_parts(Cout)
    rgb_w = torch.randn(B, 3, Cout, device=dev)
    part = torch.empty((nparts, B, 3, H, W), device=dev)

    def run():
        _cabi.call('rw_modconv_fwd_fused', _p(planes.hi), _p(planes.lo), _p(w_hi), _p(w_lo), _p(dm),
                   _p(noise), noise.stride(0), _p(nw), _p(bias), 1, B, Cin, Cout, H, W, None,
                   _p(nscale), _p(nh), _p(nl), _p(rgb_w), _p(part), _stream())
    nbytes = planes.rows * Cin * 4 + planes.rows * Cout * 4 + part.numel() * 4
    return run, flop, nbytes, '3x3 row-GEMM (next planes + ToRGB partials)'


def time_layer(run, reps, flush):
    run()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b) / 1e3
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_highres: no CUDA device')
    res = {'card': card(), 'l2_flush': 'a 512 MiB buffer is zeroed before every timed step'}
    flush = torch.empty(128 * 2 ** 20, dtype=torch.float32, device='cuda')
    models = {s: seeded(s).cuda() for s in (512, 1024)}
    rates = {}
    for size, B in ((1024, 8), (1024, 16), (512, 16)):
        r, e = gen_rate(models[size], B, args.steps, args.warmup, flush)
        rates['%d_b%d' % (size, B)] = {'img_s_resident': round(r, 2), 'img_s_e2e_u8': round(e, 2)}
    res['generator'] = rates
    layers = {}
    with torch.no_grad():
        for num in range(13, 19):
            run, flop, nbytes, kind = layer_launches(models[1024], num, 8)
            t = time_layer(run, max(args.steps, 5), flush)
            t_min = max(flop / PEAK_FLOPS, nbytes / PEAK_BYTES)
            layers['layer%d' % num] = {
                'kind': kind, 'ms': round(t * 1e3, 3), 'gflop': round(flop / 1e9, 2),
                'gbytes': round(nbytes / 1e9, 3), 'tflop_s': round(flop / t / 1e12, 1),
                'tb_s': round(nbytes / t / 1e12, 2),
                'bound': 'compute' if flop / PEAK_FLOPS >= nbytes / PEAK_BYTES else 'HBM',
                'share_of_bound': round(t_min / t, 3)}
            torch.cuda.empty_cache()
    res['layers_1024_b8'] = layers
    # the CPU oracle (fp32 torch on the host) at 512^2, one image
    from oracle import sg2_oracle as orc
    from rewriting_b200.utils import zdataset
    sd = {k: v.detach().cpu() for k, v in models[512].state_dict().items()}
    z = zdataset.standard_z_sample(1, 512, seed=3)
    t0 = time.perf_counter()
    with torch.no_grad():
        orc.generator_forward(sd, z, size=512)
    res['oracle_cpu_s_per_img_512'] = round(time.perf_counter() - t0, 2)
    res['oracle_cpu_threads'] = torch.get_num_threads()
    res['card_after'] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
