#!/usr/bin/env python
"""bench.py — headline benchmark of the rewriting_b200 hot path (driver contract).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

metric   : StyleGAN2-256 images/sec (BASELINE.json), synthetic random z, seeded random weights
workload : SeqStyleGAN2(256, mconv='seq') generator forward, batch=32 per GPU, fp32 in/out,
           conv operands 3-term split bf16 on tcgen05 tensor cores (fp32 accumulate)
step     : one batch of 32 latents through the whole generator -> 32 images (per GPU)
value    : images/s with z resident in HBM, CUDA-event timed, max over ranks, whole job
e2e      : same through the public API with HOST buffers: pinned z -> H2D, model(z), D2H of
           the images into pinned memory, inside the timed region
extra    : the other BASELINE.json configs as stated —
           config 3: key-covariance samples/sec, layer 8, 10 000 z through
             SeqStyleGanRewriter.collect_2nd_moment, STRONG scaling over the ranks, the one
             all-reduce of (mom2, count) inside the timing (also reported as `roofline_cov`);
           config 4: the shipped hat_on_horse_ears.json request, 1000 z, 2001 iterations:
             apply_edit (key finding + insert) and the insert loop alone, its/s ("replicas only");
           config 5: 50 010 images (reference batches of 10, seed 10*j) sharded over the ranks,
             uint8 NHWC out, pipelined D2H;
           config 2: fused StyledConv forward + backward over all 13 layer shapes (N = 1 only)
roofline : dominant kernel = conv_tc (implicit-GEMM styled conv); achieved = algorithmic conv
           FLOPs / summed CUDA-event kernel time, against the MEASURED bf16 tensor peak
cpu_baseline / --impl reference: the CPU oracle port of the reference's PyTorch path
           (oracle/sg2_oracle.py; the Python reference itself cannot travel to the GPU box)
           timed on the host cores on a bounded sample (batch 2).

--dump-outputs DIR: after the run, DIR/images.npy holds what the timed path returned in its last
           step: rank 0's batch of 32 images, float32 [32, 3, 256, 256] (24 MiB).  z and the
           weights are seeded, so two builds given the same arguments can be compared image
           for image.

Multi-GPU: one process per GPU under torchrun; z batches are independent (weak scaling, no
data-path collective for image generation; one all-reduce for the covariance).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def cpu_threads():
    """torch CPU convs at batch 2 stop scaling past ~16 threads (measured on the 128-core GPU
    host: 8 thr 1.11 s, 16 thr 0.96 s, 32 thr 0.98 s, 64 thr 1.41 s, 128 thr 19 s per forward),
    so the baseline uses the fastest setting, not the core count."""
    return max(1, min(os.cpu_count() or 1, 16))


# torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU-baseline legs (rank 0 only) would
# then run single-threaded inside MKL/oneDNN whatever torch.set_num_threads says later
if os.environ.get('OMP_NUM_THREADS', '1') == '1':
    os.environ['OMP_NUM_THREADS'] = str(cpu_threads())
    os.environ.setdefault('MKL_NUM_THREADS', str(cpu_threads()))

import torch  # noqa: E402

BATCH = 32
SIZE = 256
GFLOP_PER_IMG = 90.24          # algorithmic conv FLOPs of one 256^2 forward (SURVEY.md App. A)
GFLOP_PER_COV_SAMPLE = 3.71    # context forward to layer 8 + key second moment, per z (§8d)
N_COV = 10000                  # BASELINE config 3
N_SAMPLE_IMAGES = 50000        # BASELINE config 5 (the reference generates 50 010)
METRIC = 'StyleGAN2-256 images/sec'


def conv_gflop_layers():
    """Algorithmic GFLOP per image of each styled conv (up layers counted on input res)."""
    chans = {4: 512, 8: 512, 16: 512, 32: 512, 64: 512, 128: 256, 256: 128}
    out = {}
    out['layer2'] = 2 * 512 * 512 * 9 * 16 / 1e9
    n = 3
    cin = 512
    for res in (8, 16, 32, 64, 128, 256):
        cout = chans[res]
        out['layer%d' % n] = 2 * cin * cout * 9 * (res // 2) ** 2 / 1e9
        out['layer%d' % (n + 1)] = 2 * cout * cout * 9 * res ** 2 / 1e9
        n += 2
        cin = cout
    return out


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(tflops=float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1590.0))),
                    hbm=float(d.get('hbm_gbs', 6650.0)), source='measured (MEASURED_PEAKS.json, '
                    'sustained bf16 GEMM)')
    return dict(tflops=1400.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


class ClockSampler(object):
    """Polls nvidia-smi (one-shot queries from a thread: its -lms loop block-buffers when
    piped) for SM clocks and throttle reasons while the timed region runs."""
    FIELDS = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._thread = None

    def _poll(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                     '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                for ln in out.stdout.strip().splitlines():
                    self.rows.append([p.strip() for p in ln.split(',')])
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._thread = threading.Thread(target=self._poll, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=6)
        sm, mx, reasons = [], None, set()
        for parts in self.rows:
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, parts[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx,
                    reasons=sorted(reasons), samples=len(sm))


def build_model(device):
    from rewriting_b200.synthetic import seeded_generator    # the product arm imports no oracle/
    return seeded_generator(SIZE).to(device).eval()


def cpu_baseline_generator(seconds=12.0, batch=2):
    """Oracle port of the reference's generator forward on the host cores (bounded sample)."""
    from oracle import sg2_oracle as orc
    from rewriting_b200.utils.stylegan2 import SeqStyleGAN2
    from rewriting_b200.utils import zdataset
    cores = cpu_threads()
    torch.set_num_threads(cores)
    model = orc.seeded_state_dict(lambda: SeqStyleGAN2(SIZE, style_dim=512, n_mlp=8, mconv='seq'))
    sd = {k: v for k, v in model.state_dict().items()}
    z = zdataset.standard_z_sample(batch, 512, seed=1)
    with torch.no_grad():
        orc.generator_forward(sd, z)          # warm-up
        n, t0 = 0, time.time()
        while True:
            orc.generator_forward(sd, z)
            n += 1
            if time.time() - t0 > seconds or n >= 64:
                break
        dt = time.time() - t0
    out = dict(value=batch * n / dt, unit='images/s', cores=cores, kind='port',
               sample='%d forwards of batch %d (%.1f s), oracle/sg2_oracle.py generator_forward, '
                      'torch CPU fp32, %d threads' % (n, batch, dt, cores))
    # the other two quantities bench `extra` reports, on bounded samples (SURVEY.md §8d):
    # key covariance (context forward to layer 8 + second moment) and the rewrite loop
    try:
        with torch.no_grad():
            t0 = time.time()
            zc = zdataset.standard_z_sample(4, 512, seed=1)
            keys = [orc.generator_forward(sd, zc[i:i + 2], upto_key_layer=8) for i in (0, 2)]
            orc.second_moment(keys)
            dt_cov = time.time() - t0
        k = keys[0][:1, :, 10:18, 12:21].contiguous()
        style = torch.ones(1, 512)
        w = sd['layer8.sconv.mconv.dconv.weight'].clone()
        tgt = orc.target_forward(k, style, w, sd['layer8.sconv.noise.weight'],
                                 sd['layer8.sconv.activate.bias']) * 1.5 + 0.3
        q, _ = torch.linalg.qr(torch.randn(512, 1))
        its = 10
        t0 = time.time()
        orc.insert_loop(w, k, style, tgt, sd['layer8.sconv.noise.weight'],
                        sd['layer8.sconv.activate.bias'], q.t().contiguous(), its)
        dt_ins = time.time() - t0
        out['extra'] = {'key_covariance_samples_per_s': 4 / dt_cov,
                        'insert_its_per_s': its / dt_ins,
                        'sample': '4 z to layer 8 + second moment (%.1f s); %d insert iterations on '
                                  'a 1x512x8x9 key (%.1f s); same oracle port, %d threads'
                                  % (dt_cov, its, dt_ins, cores)}
    except Exception as e:  # noqa: BLE001
        out['extra'] = {'error': '%s: %s' % (type(e).__name__, e)}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU path (oracle port) on the host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    from oracle import sg2_oracle as orc
    from rewriting_b200.utils.stylegan2 import SeqStyleGAN2
    from rewriting_b200.utils import zdataset
    cores = cpu_threads()
    torch.set_num_threads(cores)
    model = orc.seeded_state_dict(lambda: SeqStyleGAN2(SIZE, style_dim=512, n_mlp=8, mconv='seq'))
    sd = dict(model.state_dict())
    sample = 2                              # images per step (bounded sample of the batch of 32)
    z = zdataset.standard_z_sample(sample, 512, seed=1)
    steps = max(1, min(args.steps, 40))
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 3))):
            orc.generator_forward(sd, z)
        t0 = time.time()
        for _ in range(steps):
            orc.generator_forward(sd, z)
        dt = time.time() - t0
    val = sample * steps / dt
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'images/s',
        'n_gpus': args.gpus, 'steps': steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * dt / steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'SeqStyleGAN2-256 generator forward (mconv=seq), seeded random '
                               'weights, random z; each step = bounded sample of %d images of '
                               'the batch-32 workload' % sample},
        'cpu_baseline': {'value': val, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d steps x %d images, oracle port of the reference PyTorch '
                                   'path (the Python reference cannot travel to the GPU box)'
                                   % (steps, sample)},
        'e2e': {'value': val, 'unit': 'images/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-extra', action='store_true', help='skip covariance / insert extras')
    ap.add_argument('--sample-images', type=int, default=N_SAMPLE_IMAGES,
                    help='images of the config-5 sampling leg (0 skips it)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true',
                    help='time eager module calls instead of the CUDA-graph replay')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the images of the last timed step to DIR/images.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)

    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the product has no CPU path)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
    W = max(args.warmup, 3)
    K = args.steps

    from rewriting_b200 import _cabi, ops
    from rewriting_b200.utils import zdataset, nethook, runningstats
    from rewriting_b200 import dist as rdist
    _cabi.load()
    model = build_model(device)

    # per-rank z shard (weak scaling: every rank gets its own K+W batches of 32)
    n_batches = W + K
    z_all = zdataset.standard_z_sample(BATCH * n_batches * world, 512, seed=1)
    z_mine = z_all[rank * BATCH * n_batches:(rank + 1) * BATCH * n_batches].contiguous()
    z_dev = z_mine.to(device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- per-kernel event timing of the dominant kernel (conv_tc) -------------------------
    # every conv_tc launch goes through one of these C-ABI entry points; bracket them with
    # CUDA events on the launching stream (argument positions: B, Cin, Cout, H, W)
    conv_events = []
    timing_on = {'on': False}
    CONV_ENTRY = {'rw_modconv_fwd': (10, 11, 12, 13, 14), 'rw_modconv_fwd_fused': (10, 11, 12, 13, 14),
                  'rw_modconv_up_fwd': (5, 6, 7, 8, 9), 'rw_modconv_up_fwd_cl': (5, 6, 7, 8, 9),
                  'rw_modconv_up_fused': (13, 14, 15, 16, 17)}
    orig_call = _cabi.call

    def timed_call(name, *a):
        if not timing_on['on'] or name not in CONV_ENTRY:
            return orig_call(name, *a)
        iB, iCi, iCo, iH, iW = CONV_ENTRY[name]
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record()
        orig_call(name, *a)
        ev1.record()
        conv_events.append((ev0, ev1, 2.0 * a[iB] * a[iCi] * a[iCo] * 9 * a[iH] * a[iW],
                            'up' if name == 'rw_modconv_up_fused' else 'conv'))
    _cabi.call = timed_call

    # ---- public API objects: eager module and its CUDA-graph replay -------------------------
    from rewriting_b200.graphs import GraphedModule
    use_graph = not args.no_graph
    with torch.no_grad():
        model(z_dev[:BATCH])                               # one-off weight-plane preparation
        launches0 = _cabi.launch_count
        model(z_dev[:BATCH])
    launches_per_step = _cabi.launch_count - launches0     # kernels of ONE forward (mine only)
    runner = GraphedModule(model, z_dev[:BATCH]) if use_graph else model

    # ---- device-resident timing ------------------------------------------------------------
    with torch.no_grad():
        for i in range(W):
            runner(z_dev[i * BATCH:(i + 1) * BATCH])
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(W, W + K):
            flush.zero_()                                        # evict L2 between steps
            img = runner(z_dev[i * BATCH:(i + 1) * BATCH])
        e1.record()
        barrier()
        ms_dev = max_over_ranks(e0.elapsed_time(e1))
        # the graph replay returns its static output buffer, which later replays overwrite
        last_images = img.float().cpu() if args.dump_outputs and rank == 0 else None
        launches = launches_per_step * K          # a graph replay launches the same kernels
        # per-kernel CUDA-event timing of the dominant kernel: eager replay of the same steps
        # (events cannot be read back from inside a graph), CPU running ahead of the GPU
        for i in range(2):
            model(z_dev[i * BATCH:(i + 1) * BATCH])
        torch.cuda.synchronize()
        timing_on['on'] = True
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(W, W + K):
            flush.zero_()
            model(z_dev[i * BATCH:(i + 1) * BATCH])
        t1.record()
        torch.cuda.synchronize()
        timing_on['on'] = False
        ms_eager = t0.elapsed_time(t1)
    # dominant kernel = conv_tc (the 3x3 styled convs); the fused upsampling kernel
    # (conv_transpose + blur + activation in one launch) is reported next to it
    conv_ms = sum(a.elapsed_time(b) for a, b, _, k in conv_events if k == 'conv')
    conv_flops = sum(f for _, _, f, k in conv_events if k == 'conv')
    conv_launches = sum(1 for _, _, _, k in conv_events if k == 'conv')
    up_ms = sum(a.elapsed_time(b) for a, b, _, k in conv_events if k == 'up')
    up_flops = sum(f for _, _, f, k in conv_events if k == 'up')
    up_launches = sum(1 for _, _, _, k in conv_events if k == 'up')
    conv_events.clear()

    # ---- end-to-end timing through the public API with host buffers ------------------------
    z_host = z_mine.pin_memory()
    out_host = torch.empty(BATCH, 3, SIZE, SIZE).pin_memory()
    out_hosts = [out_host, torch.empty(BATCH, 3, SIZE, SIZE).pin_memory()]
    with torch.no_grad():
        runner(z_host[:BATCH].to(device, non_blocking=True))
        barrier()
        s0 = torch.cuda.Event(enable_timing=True)
        s1 = torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(W, W + K):
            flush.zero_()
            if use_graph:       # pinned z -> static input (H2D), replay, images -> pinned host
                runner(z_host[i * BATCH:(i + 1) * BATCH], out=out_hosts[i & 1])
            else:
                zb = z_host[i * BATCH:(i + 1) * BATCH].to(device, non_blocking=True)
                out_host.copy_(model(zb), non_blocking=True)
        if use_graph:
            # the timed region ends when the LAST image batch has landed in host memory
            torch.cuda.current_stream().wait_stream(runner._copy_stream)
        s1.record()
        barrier()
        ms_e2e = max_over_ranks(s0.elapsed_time(s1))
    # SM clocks / throttle reasons sampled over all three timed loops (device-resident, per-kernel
    # replay, end-to-end): the first alone lasts ~0.2 s, i.e. one or two nvidia-smi polls
    clocks = sampler.stop() if rank == 0 else None

    value = BATCH * K * world / (ms_dev / 1e3)
    e2e_value = BATCH * K * world / (ms_e2e / 1e3)

    # ---- extras: BASELINE configs 3, 4, 5 as stated, and config 2 --------------------------
    extra = {}
    cov = None
    if not args.no_extra:
        del runner
        torch.cuda.empty_cache()
        try:
            cov = bench_config3(model, device, world, rank, barrier, max_over_ranks)
            extra['config3_key_covariance'] = cov
            extra['key_covariance_samples_per_s'] = cov['samples_per_s']
        except Exception as e:  # noqa: BLE001
            extra['config3_key_covariance'] = {'error': '%s: %s' % (type(e).__name__, e)}
        try:
            extra['config4_rewrite'] = bench_config4(model, device)
        except Exception as e:  # noqa: BLE001
            extra['config4_rewrite'] = {'error': '%s: %s' % (type(e).__name__, e)}
        try:
            extra['config5_sampling'] = bench_config5(model, device, world, barrier, max_over_ranks,
                                                      args.sample_images)
        except Exception as e:  # noqa: BLE001
            extra['config5_sampling'] = {'error': '%s: %s' % (type(e).__name__, e)}
        if world == 1:
            # BASELINE.json configs[1]: fused StyledConv forward + backward (dX, dstyle, dW, dbias,
            # dnoise), every layer shape of the 256^2 generator at batch 32
            try:
                torch.cuda.empty_cache()
                from tools import bench_modconv
                r = bench_modconv.main(B=BATCH, quiet=True, save=False)
                sm = r['summary']
                extra['modconv_fwdbwd_b32'] = {
                    'fwd_ms': sm['total_fwd_ms'], 'fwdbwd_ms': sm['total_fwdbwd_ms'],
                    'fwd_TFLOPs': sm['fwd_TFLOPs'], 'fwdbwd_TFLOPs': sm['fwdbwd_TFLOPs'],
                    'per_layer_fwdbwd_ms': {l['layer']: round(l['fwdbwd_ms'], 4) for l in r['layers']},
                    'note': sm['note']}
            except Exception as e:  # noqa: BLE001
                extra['modconv_fwdbwd_b32'] = {'error': '%s: %s' % (type(e).__name__, e)}

    if rank == 0:
        peaks = measured_peaks()
        # DRAM bytes per launch of the dominant kernel class: ncu (dram__bytes_read.sum +
        # dram__bytes_write.sum) over every conv launch of one forward of THIS command, digested
        # by tools/dram_summary.py into profiles/ (a profiler cannot run inside the timed bench)
        traffic, traffic_note = None, None
        prof = os.path.join(ROOT, 'profiles', 'r2_dram_per_launch.json')
        if os.path.exists(prof):
            try:
                with open(prof) as f:
                    dj = json.load(f)
                ent = dj['kernels']['conv (conv_tc + upconv_fused)']
                traffic = ent['dram_bytes_per_launch']
                traffic_note = ('mean over the %d styled-conv launches of one forward, %s; '
                                'algorithmic bytes per launch %.3g' % (
                                    ent['launches'], dj['source'], ent['algorithmic_bytes_per_launch']))
            except Exception:
                traffic = None
        achieved = (conv_flops / 1e12) / (conv_ms / 1e3) if conv_ms > 0 else 0.0
        line = {
            'metric': METRIC, 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': K,
            'warmup': W, 'ms_per_step': ms_dev / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None,
            'dtype': 'bf16x3 (3-term split bf16 operands, fp32 accumulate; fp32 in/out)',
            'data': 'synthetic',
            'config': {'workload': 'SeqStyleGAN2-256 (mconv=seq, channel_multiplier=2) generator '
                                   'forward, batch=%d per GPU, seeded random weights, random z '
                                   '(zdataset seed 1)' % BATCH,
                       'execution': 'CUDA graph replay of model(z) (rewriting_b200.graphs.'
                                    'GraphedModule)' if use_graph else 'eager model(z)',
                       'global_batch': BATCH * world, 'parallelism': 'dp%d (independent z shards)'
                       % world, 'l2': 'flushed between steps (256 MiB memset, inside the timed region)',
                       'gflop_per_image': GFLOP_PER_IMG},
            'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peaks['tflops'],
                         'unit': 'TFLOP/s', 'frac': achieved / peaks['tflops'],
                         'traffic': traffic, 'traffic_source': traffic_note,
                         'kernel': 'rw::conv_tc_kernel<128> (the 3x3 styled-conv launches of the '
                         'timed steps: layers 2,4,...,14)', 'kernel_launches': conv_launches,
                         'kernel_ms_per_step': conv_ms / K,
                         'kernel_share_of_step': (conv_ms / K) / (ms_eager / K),
                         'timed_in': 'eager replay of the timed steps (%.2f ms/step); the headline '
                                     'value is the %s' % (ms_eager / K, 'CUDA-graph replay of the '
                                     'same module call' if use_graph else 'eager call'),
                         'peak_source': peaks['source'],
                         'note': 'algorithmic FLOPs (1x) against the cuBLAS-measured sustained bf16 '
                                 'peak; the 3-term split issues 3x the MMAs, so frac ~ 1/3 means the '
                                 'tensor pipe is as busy as in a cuBLAS GEMM; tensor-pipe utilisation '
                                 'per layer is in profiles/'},
            'e2e': {'value': e2e_value, 'unit': 'images/s', 'ms_per_step': ms_e2e / K,
                    'h2d_bytes_per_step': BATCH * 512 * 4,
                    'd2h_bytes_per_step': BATCH * 3 * SIZE * SIZE * 4},
            'gpu_launches': launches,
            'clocks': clocks,
            'extra': extra,
        }
        if up_ms > 0:
            up_tf = (up_flops / 1e12) / (up_ms / 1e3)
            line['roofline_upconv'] = {
                'bound': 'tensor', 'achieved': up_tf, 'peak': peaks['tflops'], 'unit': 'TFLOP/s',
                'frac': up_tf / peaks['tflops'], 'kernel': 'rw::upconv_fused_kernel (layers 3,5,...,13: '
                'conv_transpose + 4x4 blur + demod + noise + bias + leaky-ReLU + next-layer planes in one '
                'launch; FLOPs counted for the conv_transpose only)', 'kernel_launches': up_launches,
                'kernel_ms_per_step': up_ms / K,
                'note': 'layer 13 is epilogue-bound (SIMT FIR + activation behind the MMAs: 5.2k cycles '
                        'per row step against 3.7k of MMAs), layers 9/11 wait for the MMAs half of the '
                        'time (3-term split: frac <= 1/3), tools/prof_upconv.py + DESIGN.md §6; the '
                        'round-1 pair (conv_transpose GEMM + SIMT blur) moved 2.3x the DRAM bytes of the '
                        'layer pair'}
        if cov is not None and 'samples_per_s' in cov:
            # second half of BASELINE.json's metric: key-covariance samples/s (config 3)
            cov_tf = cov['samples_per_s'] * GFLOP_PER_COV_SAMPLE / 1e3
            line['roofline_cov'] = {
                'bound': 'tensor', 'achieved': cov_tf, 'peak': peaks['tflops'] * world,
                'unit': 'TFLOP/s', 'frac': cov_tf / (peaks['tflops'] * world),
                'flop_per_unit': '%.2f GFLOP per z: context forward to layer 8 (3.17) + 1024 x '
                                 '512^2 second moment (0.54), SURVEY.md §8d' % GFLOP_PER_COV_SAMPLE,
                'kernels': 'conv_tc / upconv_fused (layers 2-7) + gram_tc, whole collection '
                           'incl. the all-reduce', 'peak_source': peaks['source']}
        if not args.no_cpu_baseline and world == 1:
            line['cpu_baseline'] = cpu_baseline_generator()
        elif world > 1:
            line['cpu_baseline'] = {'value': None, 'unit': 'images/s', 'cores': os.cpu_count(),
                                    'kind': 'port', 'sample': 'measured at N=1 only'}
        if last_images is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, 'images.npy'), last_images.numpy())
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def bench_config3(model, device, world, rank, barrier, max_over_ranks, repeats=3):
    """BASELINE config 3 as stated: layer-8 key covariance C over 10 000 random z through
    `SeqStyleGanRewriter.collect_2nd_moment` (reference ganrewrite.py:83-96, tally.py:424-443),
    STRONG scaling: the 10 000 z are sharded over the ranks, one all-reduce of (mom2, count)
    inside the timed region, every rank ends with the same matrix."""
    from rewriting_b200.rewrite import ganrewrite
    from rewriting_b200.utils import zdataset
    zds = torch.utils.data.TensorDataset(zdataset.standard_z_sample(N_COV, 512, seed=1))
    # the constructor runs one full collection: graph capture + weight planes = warm-up
    gw = ganrewrite.SeqStyleGanRewriter(model, zds, 8)
    c_first = gw.c_matrix.clone()
    times = []
    for _ in range(repeats):
        barrier()
        t0 = time.perf_counter()
        C = gw.collect_2nd_moment()
        torch.cuda.synchronize()
        times.append(max_over_ranks((time.perf_counter() - t0) * 1e3))
    ms = sorted(times)[len(times) // 2]
    rel = float(((C.to(device) - c_first).norm() / c_first.norm()).item())
    return {'n_z': N_COV, 'layer': 8, 'scaling': 'strong', 'ms_total': ms,
            'samples_per_s': N_COV / (ms / 1e3), 'ms_all_repeats': times,
            'pass_size': gw._moment_bs, 'passes_per_rank': -(-N_COV // (gw._moment_bs * world)),
            'repeatability_rel_fro': rel,
            'timing': 'host clock around collect_2nd_moment() between device synchronisations '
                      '(the call ends with C on the host), max over ranks, median of %d' % repeats,
            'collective': 'one all_reduce(sum) of mom2[512,512] fp32 + count, inside the timing'}


def bench_config4(model, device):
    """BASELINE config 4 as stated: rank-1 projected-gradient rewrite on the shipped request
    notebooks/masks/stylegan/horse/hat_on_horse_ears.json (committed copy under tests/golden/),
    4 context keys, zds = 1000, layer 8, 2001 iterations, piter 10, lr 0.05 — through
    `apply_edit` (key finding + insert) and the insert loop alone (ganrewrite.py:135-169, 254-298)."""
    from rewriting_b200.rewrite import ganrewrite
    from rewriting_b200.utils import zdataset
    with open(os.path.join(ROOT, 'tests', 'golden', 'hat_on_horse_ears.json')) as f:
        request = json.load(f)
    zds = torch.utils.data.TensorDataset(zdataset.standard_z_sample(1000, 512, seed=1))
    t0 = time.perf_counter()
    gw = ganrewrite.SeqStyleGanRewriter(model, zds, 8)
    torch.cuda.synchronize()
    t_init = time.perf_counter() - t0
    W0 = gw.target_weights().detach().clone()

    def restore():
        with torch.no_grad():
            gw.target_weights()[...] = W0
    gw.apply_edit(request, rank=1, niter=50)                     # warm-up (graphs, caches)
    restore()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gw.apply_edit(request, rank=1, niter=2001, piter=10, lr=0.05)
    torch.cuda.synchronize()
    t_edit = time.perf_counter() - t0
    restore()
    with torch.no_grad():
        obj_acts, _, obj_area, _ = gw.object_from_selection(*request['object'])
        goal_in, goal_out, _, _ = gw.paste_from_selection(request['paste'][0], request['paste'][1],
                                                          obj_acts, obj_area)
        d = gw.multi_key_from_selection(request['key'], rank=1)
    losses = []
    ms = gw.insert(goal_in, goal_out, d, niter=2001, piter=10, lr=0.05, return_timing=True)
    restore()
    gw.insert(goal_in, goal_out, d, niter=2001, piter=10, lr=0.05,
              update_callback=lambda it, loss: losses.append(loss))
    restore()
    crop = list(goal_in.fmap.shape)
    Cout, Cin = W0.shape[1], W0.shape[2]
    P = crop[0] * crop[2] * crop[3]
    flop_it = 2.0 * 2 * P * Cout * Cin * 9            # forward conv on the crop + weight gradient
    state_bytes = 6 * Cout * Cin * 9 * 4              # W, m, v read + written if they streamed from HBM
    key_bytes = 2 * (Cout // 4) * crop[0] * (crop[2] + 2) * (crop[3] + 2) * Cin * 4
    its = 2001 / (ms / 1e3)
    return {'request': 'hat_on_horse_ears.json (object 441, paste 854, keys 354/956/309/926)',
            'niter': 2001, 'rank': 1, 'key_crop': crop, 'rewriter_init_s_1000z': t_init,
            'apply_edit_s': t_edit, 'apply_edit_its_per_s': 2001 / t_edit,
            'insert_ms': ms, 'insert_its_per_s': its,
            'final_loss': float(losses[-1]), 'first_loss': float(losses[0]),
            'roofline': {
                'bound': 'latency (neither L2 nor HBM bandwidth)',
                'l2_key_traffic_GBps': key_bytes * its / 1e9,
                'fp32_TFLOPs': flop_it * its / 1e12,
                'hbm_equivalent_GBps_if_state_streamed': state_bytes * its / 1e9,
                'note': 'W[o] lives in shared memory for all iterations, m/v stream through L2; '
                        'the key crop is re-read from L2 by every 4-channel CTA twice per iteration. '
                        'ncu (profiles/r2_ncu_insert_before_details.txt): DRAM 0.03 %, L2 3.8 %, L2 hit '
                        '99.4 %, issue slots 46 %, 8 warps/SM at 255 registers: latency-bound '
                        '(stall_wait / long_scoreboard on the L2 key loads), 128 of 148 SMs busy '
                        '(512 output channels / 4 per CTA)'}}


def bench_config5(model, device, world, barrier, max_over_ranks, nimgs):
    """BASELINE config 5: 50 000-sample generation (the reference generates 50 010:
    utils/get_samples.py:114-129), reference batches of 10 with seed 10*j sharded over the ranks,
    uint8 NHWC written by the last ToRGB combine, pipelined D2H into pinned host memory."""
    if nimgs <= 0:
        return {'skipped': True}
    from rewriting_b200 import sampling
    seen = {'n': 0, 'sum': 0}

    def sink(images, batches):
        seen['n'] += images.shape[0]
        seen['sum'] += int(images[0, 0, 0, 0])            # touch the landed data
    sampling.get_samples(model, nimgs=640 * world, out_dtype=torch.uint8, group=4,
                         sink=lambda im, b: None)              # warm-up: capture + pinned ring
    barrier()
    t0 = time.perf_counter()
    _, mine = sampling.get_samples(model, nimgs=nimgs, out_dtype=torch.uint8, group=4, sink=sink)
    torch.cuda.synchronize()
    ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    total = (nimgs // 10 + 1) * 10
    return {'images': total, 'ms_total': ms, 'images_per_s': total / (ms / 1e3),
            'this_rank_images': seen['n'], 'images_per_replay': 40, 'out': 'uint8 NHWC on the host',
            'd2h_bytes': total * SIZE * SIZE * 3, 'scaling': 'strong',
            'timing': 'host clock around get_samples() incl. z generation, H2D, D2H; max over ranks'}


if __name__ == '__main__':
    sys.exit(main())
