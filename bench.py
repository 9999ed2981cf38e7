#!/usr/bin/env python
"""bench.py — images/sec at fixed NFE for the BASELINE headline configuration.

    python bench.py --gpus N --steps K --warmup W            # native arm (one process per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path, timed on the host cores (rank 0 only)
    python bench.py ... --dump-outputs DIR                   # also write the samples of the last timed step to DIR/*.npy

Workload (BASELINE.json configs[1]): EDM CIFAR-10 32x32 DDPM++ U-Net (random init, de-zeroed so |F_x| = O(1)), Heun sampler,
num_steps=10 => NFE=18, batch 512 per GPU, synthetic Gaussian latents.  One "step" = one full sampling pass over one batch.
`value` = images/sec with latents resident in HBM; `e2e` = the same through the public API with pinned-host latents copied in
and finished images copied back every step.  Scaling is weak: every rank samples its own 512-image batch, no collective on
the sampling path; one NCCL all_gather of the uint8 images after the timed region (what FID consumes).

At N=1 the same line also carries (rank 0, after the headline measurement; `--no_extras` skips them):
  `configs`    BASELINE configs 3, 4 and 5 (FFHQ-64 iPNDM NFE=6, ImageNet-64 DPM-Solver++(2M) NFE=10, SD-v1.5 AMED-DPM++ NFE=5) measured the
               same way (value, e2e, roofline, precision) at their per-GPU batch, >= 10 timed steps each;
  `gpu_eager`  the reference's own GPU path -- eager PyTorch (cuDNN / cuBLAS: F.conv2d, F.group_norm, einsum attention), stated through the
               functional nets of oracle/ (bit-identical to the reference modules on CPU, tests/golden) -- on the same B200, same batch / NFE:
               the "beat PyTorch-eager on the same GPU" bar of SURVEY.md section 2.2.  A comparator, never the thing measured as `value`.
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

GFLOP_PER_IMG_NFE = {'cifar10': 42.38, 'ffhq': 83.73, 'imagenet64': 219.33, 'sd15': 2 * 803.27}      # BASELINE.md section 2 (2 FLOP per MAC; SD: x2 under CFG)
SOLVER_NFE = {'heun': lambda n: 2 * (n - 1), 'euler': lambda n: n - 1, 'ipndm': lambda n: n - 1, 'dpm_pp': lambda n: n - 1,
              'amed_dpm_pp': lambda n: 2 * (n - 1) - 1}      # AMED plug-in with AFS: num_steps=4 -> NFE=5 (amed-solver-main/README.md)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--net', default='cifar10', help='cifar10 | ffhq | imagenet64 | sd15')
    ap.add_argument('--solver', default='heun', help='heun | euler | ipndm | dpm_pp | amed_dpm_pp (sd15)')
    ap.add_argument('--num_steps', type=int, default=10)
    ap.add_argument('--batch', type=int, default=512, help='images per GPU per step')
    ap.add_argument('--precision', default='auto', choices=['auto', 'fp16x3', 'fp16', 'fp16f8'],
                    help="fp16x3: 3 fp16 MMAs per product; fp16f8: fp16 hi x hi + two e4m3 correction MMAs (block / head convolutions); fp16: single "
                         "pass; auto (default): the fastest mode whose final images stay within the 1e-3 contract for the named net (PRECISION_FOR)")
    ap.add_argument('--f8_min_channels', type=int, default=0, help='fp16f8 only: blocks with fewer input or output channels stay fp16x3 (0 = all blocks in f8)')
    ap.add_argument('--cpu_batch', type=int, default=8, help='batch of the bounded CPU-baseline sample')
    ap.add_argument('--no_cpu_baseline', action='store_true')
    ap.add_argument('--fuse_stats', type=int, default=1, help='1 (default): GroupNorm statistics from the GEMM epilogues; 0: separate gn_stats pass')
    ap.add_argument('--no_extras', action='store_true', help='skip the roofline / e2e / fp16 legs (timing of the main leg is unchanged)')
    ap.add_argument('--all_configs', type=int, default=1, help='1 (default, N=1 only): also measure BASELINE configs 3-5 into `configs`')
    ap.add_argument('--config_steps', type=int, default=10, help='timed steps of each `configs` entry')
    ap.add_argument('--gpu_eager', type=int, default=1, help='1 (default, N=1 only): time the eager-PyTorch GPU path of the same configs')
    ap.add_argument('--dump-outputs', dest='dump_outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned (rank 0; each `configs` entry too) as DIR/<name>.npy in '
                         f'float32, at most {DUMP_LIMIT_BYTES >> 20} MB in all')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.precision_requested = args.precision
    args.f8_min_channels_requested = args.f8_min_channels
    if args.precision == 'auto':
        args.precision = PRECISION_FOR.get(args.net, 'fp16x3')
        if args.f8_min_channels == 0:
            args.f8_min_channels = F8_MIN_CHANNELS_FOR.get(args.net, 0)
    return args


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d['hbm_gbs'], tflops_burst=d['bf16_tflops'], tflops_sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, arrays):
    """`--dump-outputs`: every {name: tensor} as out_dir/<name>.npy in float32.  A run's inputs depend only on its arguments, so two builds
    run with the same arguments can be compared file by file.  Over DUMP_LIMIT_BYTES in all, every array keeps the same fraction of its
    leading (batch) rows, picked with a fixed seed, so the sample too is the same from run to run."""
    import numpy as np
    import torch
    total = sum(t.numel() * 4 for t in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().to('cpu', torch.float32)
        if total > DUMP_LIMIT_BYTES:
            keep = t.shape[0] * DUMP_LIMIT_BYTES // total
            t = t[torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
        np.save(os.path.join(out_dir, name + '.npy'), t.numpy())


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '200', '-i', str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return dict(sm_mhz=med, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_leg(args, steps, warmup):
    """The reference's CPU path on the host cores: the oracle port of solvers.<solver>_sampler on EDMPrecond (oracle/ is pinned
    bit-exact to /root/reference by tests/golden; /root/reference itself does not exist on the GPU box).  Bounded sample:
    the same net / solver / NFE on a batch of `cpu_batch` images."""
    import torch
    from oracle import edm_oracle as O
    from oracle import solvers_oracle as SO
    # thread count: measured on the B200 host (profiles/cpu_thread_sweep.py, 128 logical CPUs): one CIFAR-net forward at batch 8
    # takes 0.21 s with 16 threads, 0.27 s with 32, 0.59 s with 64 and 4.6 s with 128 (oversubscription), so the baseline uses
    # the fastest setting rather than every logical CPU.
    cores = min(os.cpu_count() or 1, int(os.environ.get('DSB_CPU_THREADS', '16')))
    torch.set_num_threads(cores)
    P, S = O.make_net(args.net, seed=0, dezero=True)
    net = O.OracleNet(P, S)
    lat = O.stacked_randn(range(args.cpu_batch), (S['img_channels'], S['img_resolution'], S['img_resolution']))
    lab = None
    if S['label_dim']:
        lab = torch.eye(S['label_dim'])[torch.arange(args.cpu_batch) % S['label_dim']]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        samples = SO.sample(net, lat, args.solver, class_labels=lab, num_steps=args.num_steps)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return dict(value=args.cpu_batch * len(times) / tot, seconds_per_step=tot / len(times), cores=cores, samples=samples,
                sample=f'{args.net} {args.solver} num_steps={args.num_steps} batch {args.cpu_batch} (same net/solver/NFE, bounded batch), '
                       f'{len(times)} timed + {warmup} warm-up passes, torch CPU fp32 {torch.__version__}, {cores} threads')


def make_config(args, world):
    nfe = SOLVER_NFE[args.solver](args.num_steps)
    return dict(workload=f'EDM {args.net} U-Net, {args.solver} num_steps={args.num_steps} (NFE={nfe}), batch {args.batch}/GPU',
                net=args.net, solver=args.solver, nfe=nfe, batch_per_gpu=args.batch, global_batch=args.batch * max(world, 1),
                weights='random init (reference constructors, seed 0), init_zero layers de-zeroed', parallelism=f'dp{world}',
                l2='per-forward activation working set (GBs) >> 126 MB L2')


def build_workload(args, dev, rank):
    """(net, sampler, kwargs, latents, labels) of one configuration."""
    import torch
    from diff_sampler_b200 import solvers
    from diff_sampler_b200.net import B200Net
    B = args.batch
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    labels = None
    if args.net == 'sd15':
        net, sampler, kw = build_sd15(args, dev, B, gen)
    else:
        net = B200Net.from_config(args.net, seed=0, dezero=True, precision=args.precision, device=dev, fuse_stats=bool(args.fuse_stats),
                                  f8_min_channels=args.f8_min_channels)
        sampler = getattr(solvers, args.solver + '_sampler')
    shape = (B, net.img_channels, net.img_resolution, net.img_resolution)
    latents = torch.randn(shape, generator=gen, device=dev)
    if args.net != 'sd15':
        if net.label_dim:
            labels = torch.eye(net.label_dim, device=dev)[torch.randint(net.label_dim, (B,), generator=gen, device=dev)]
        kw = dict(class_labels=labels, num_steps=args.num_steps, sigma_min=0.002, sigma_max=80, schedule_type='polynomial', schedule_rho=7)
    return net, sampler, kw, latents, labels


def timed_steps(fn, steps, barrier, dev, world):
    """EXACTLY `steps` calls of fn between CUDA events on the current stream, barrier + synchronize on both sides, max over ranks (ms)."""
    import torch
    import torch.distributed as dist
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for _ in range(steps):
        out = fn()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item(), out


def measure_e2e(sampler, net, kw, shape, steps, barrier, dev, world):
    """The same metric through the public sampler API with HOST buffers: pinned latents copied in and finished images copied back
    inside the timed region, every step."""
    import torch
    host_in = torch.randn(shape).pin_memory()
    host_out = torch.empty(shape).pin_memory()
    dev_in = torch.empty(shape, device=dev)

    def e2e_step():
        dev_in.copy_(host_in, non_blocking=True)
        out = sampler(net, dev_in, **kw)
        host_out.copy_(out, non_blocking=True)
    for _ in range(2):
        e2e_step()
    ms, _ = timed_steps(e2e_step, steps, barrier, dev, world)
    nbytes = host_in.numel() * 4
    return dict(value=world * shape[0] * steps / (ms / 1e3), unit='images/s', h2d_bytes_per_step=nbytes, d2h_bytes_per_step=nbytes)


def main():
    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    config = make_config(args, world)
    metric = 'images/sec at fixed NFE'

    if args.impl == 'reference':
        if rank != 0:
            return
        cb = cpu_reference_leg(args, args.steps, min(args.warmup, 1))
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dict(samples=cb['samples']))
        # same net / solver / NFE as the native arm's config; each step is a BOUNDED SAMPLE of it (batch `cpu_batch`, not batch_per_gpu)
        config['workload'] += f' -- CPU arm: each step is a bounded sample of this workload, batch {args.cpu_batch} on {cb["cores"]} host threads'
        config['sample_batch'] = args.cpu_batch
        line = dict(metric=metric, value=cb['value'], unit='images/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                    ms_per_step=cb['seconds_per_step'] * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                    data='synthetic', impl='reference', config=config,
                    cpu_baseline=dict(value=cb['value'], unit='images/s', cores=cb['cores'], kind='port', sample=cb['sample']),
                    e2e=dict(value=cb['value'], unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from diff_sampler_b200 import solver_utils
    assert torch.cuda.is_available(), 'the native arm needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # NCCL prints its version banner on stdout at communicator creation; stdout must carry exactly one JSON line.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    B = args.batch
    net, sampler, kw, latents, labels = build_workload(args, dev, rank)
    shape = tuple(latents.shape)

    def run_step():
        return sampler(net, latents, **kw)

    for _ in range(args.warmup):
        run_step()
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = net.total_launches + solver_utils.LAUNCHES[0]
    ms, images = timed_steps(run_step, args.steps, barrier, dev, world)
    launches = net.total_launches + solver_utils.LAUNCHES[0] - l0
    clk = clocks.stop() if rank == 0 else None
    value = world * B * args.steps / (ms / 1e3)
    dumps = dict(samples=images.cpu()) if args.dump_outputs and rank == 0 else None

    # ---- end-to-end through the public API with host buffers -------------------------------------------------------
    e2e = None
    if not args.no_extras:
        e2e = measure_e2e(sampler, net, kw, shape, args.steps, barrier, dev, world)

    # ---- finished samples: FID statistics path over NCCL (outside the timed region) ------------------------------------
    gathered = None
    fid_allreduce = None
    gits_nccl = None
    if world > 1:
        from diff_sampler_b200 import dist_utils, fid_stats
        u8 = dist_utils.to_uint8_nhwc(images)
        allimg = [torch.empty_like(u8) for _ in range(world)]
        dist.all_gather(allimg, u8)
        gathered = sum(x.numel() for x in allimg)
        try:
            # fid.py:61-75: per-rank feature moments, all_reduce of mu / sigma over NCCL.  Features here are the image pixels pooled to 8x8
            # (the detector is caller-supplied in the reference; what is exercised is the accumulation + collective).
            det = lambda u8: torch.nn.functional.adaptive_avg_pool2d(u8.float(), 8).flatten(1)
            st = fid_stats.FeatureStats().append_images(u8, det).reduce()
            mu, sigma = st.finalize()
            fid_allreduce = dict(features=int(mu.shape[0]), n=int(st.n), mu_norm=float((mu ** 2).sum() ** 0.5), sigma_trace=float(sigma.trace()),
                                 backend='nccl', note='fid.py:61-79 moments + all_reduce over NCCL; pooled-pixel features stand in for the caller-supplied detector')
        except Exception as e:                   # diagnostic only
            fid_allreduce = dict(error=repr(e))
        gits_nccl = None
        if args.net != 'sd15':
            try:
                # GITS schedule search with its cost-matrix all_reduce over NCCL (gits-main/gits_utils.py:134): every rank runs teacher
                # trajectories on its own latents, the [N_tea, N_tea] cost matrix is summed across ranks, all ranks get the same index list
                from diff_sampler_b200 import gits_utils
                gk = dict(dataset_name=args.net, num_warmup=4 * world, max_batch_size=4 * world, sigma_min=0.002, sigma_max=80, num_steps=6,
                          num_steps_tea=21, schedule_type='polynomial', schedule_rho=7, afs=False, metric='dev', coeff=1.15, model_source='edm',
                          solver='euler', solver_tea='euler', max_order=2, deis_mode='tab', prompt=None, guidance_rate=1.0)
                dp_list = [int(v) for v in gits_utils.get_dp_list(net, dev, **gk)]
                same = torch.tensor(dp_list, device=dev)
                lo, hi = same.clone(), same.clone()
                dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                dist.all_reduce(hi, op=dist.ReduceOp.MAX)
                gits_nccl = dict(dp_list=dp_list, identical_on_all_ranks=bool(torch.equal(lo, hi)), ranks=world, backend='nccl')
            except Exception as e:
                gits_nccl = dict(error=repr(e))

    if rank != 0:
        if world > 1:
            dist.barrier()                       # stay alive until rank 0 has finished its single-GPU diagnostic legs
            dist.destroy_process_group()
        return

    pk = peaks()
    line = dict(metric=metric, value=value, unit='images/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype=DTYPE_TEXT(args.precision), data='synthetic', config=config, gpu_launches=launches, clocks=clk, precision=args.precision,
                precision_requested=args.precision_requested, f8_min_channels=args.f8_min_channels)
    if e2e:
        line['e2e'] = e2e
    if gathered:
        line['allgather_bytes'] = gathered
    if fid_allreduce:
        line['fid_allreduce'] = fid_allreduce
    if gits_nccl:
        line['gits_nccl'] = gits_nccl

    try:
        if not args.no_extras:
            extras(args, line, net, sampler, kw, latents, labels, images, B, dev, pk)
    except Exception as e:                       # the main measurement above is already complete; report instead of dying
        line['extras_error'] = repr(e)

    solo = world == 1 and not args.no_extras
    if solo and args.gpu_eager and args.net != 'sd15':
        try:
            line['gpu_eager'] = gpu_eager_leg(args, dev, native_value=value)
        except Exception as e:
            line['gpu_eager'] = dict(error=repr(e))
    if solo and args.all_configs and (args.net, args.solver) == ('cifar10', 'heun'):
        del net, images
        torch.cuda.empty_cache()
        line['configs'] = other_configs(args, dev, pk, dumps)

    if not args.no_cpu_baseline and world == 1:
        cb = cpu_reference_leg(args, 1, 1)
        line['cpu_baseline'] = dict(value=cb['value'], unit='images/s', cores=cb['cores'], kind='port', sample=cb['sample'])
    if dumps:
        write_outputs(args.dump_outputs, dumps)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def DTYPE_TEXT(precision):
    return 'fp16 operands, fp32 accumulate' + {'fp16x3': ' (split-precision: 3 tcgen05 MMAs per product)',
                                               'fp16f8': ' (split-precision: fp16 hi x hi + two e4m3 correction MMAs per product)'}.get(precision, '')


# BASELINE.json configs[2..4] at their per-GPU batch (1024 / 4, 2048 / 8, 64 / 8 images per GPU)
OTHER_CONFIGS = [
    dict(id=3, net='ffhq', solver='ipndm', num_steps=7, batch=256, baseline='EDM FFHQ-64, iPNDM NFE=6 (4-term multistep history), batch 1024 on 4xB200'),
    dict(id=4, net='imagenet64', solver='dpm_pp', num_steps=11, batch=256,
         baseline='EDM ImageNet-64 class-cond, DPM-Solver++(2M) NFE=10 with GITS schedule, batch 2048 on 8xB200'),
    dict(id=5, net='sd15', solver='amed_dpm_pp', num_steps=4, batch=8, baseline='Stable Diffusion v1.5 latent 512x512, AMED-plugin on DPM++ NFE=5, batch 64 on 8xB200'),
]


def other_configs(args, dev, pk, dumps=None):
    """BASELINE configs 3-5 on one GPU at their per-GPU batch: value (latents resident), e2e (host buffers), roofline of the GEMM
    kernel (CUDA events per op), the eager-PyTorch comparator where the oracle has a GPU-capable net (configs 3, 4).  With `dumps`,
    each config's last timed samples go in as config<id>_samples."""
    import copy
    import torch
    out = []
    for c in OTHER_CONFIGS:
        a = copy.copy(args)
        a.net, a.solver, a.num_steps, a.batch = c['net'], c['solver'], c['num_steps'], c['batch']
        a.precision = PRECISION_FOR.get(a.net, 'fp16x3') if args.precision_requested == 'auto' else args.precision
        a.f8_min_channels = F8_MIN_CHANNELS_FOR.get(a.net, 0) if a.precision == 'fp16f8' else 0
        ent = dict(id=c['id'], baseline_config=c['baseline'], workload=make_config(a, 1)['workload'], precision=a.precision,
                   f8_min_channels=a.f8_min_channels, steps=args.config_steps)
        try:
            t0 = time.time()
            net, sampler, kw, latents, labels = build_workload(a, dev, 0)
            if a.solver == 'dpm_pp' and a.net == 'imagenet64':
                # config 4 samples on a GITS schedule: 11 of the 61 teacher grid points, picked by the DP over native teacher trajectories
                from diff_sampler_b200 import gits_utils, solver_utils
                gk = dict(dataset_name='imagenet64', num_warmup=16, max_batch_size=16, sigma_min=0.002, sigma_max=80, num_steps=11, num_steps_tea=61,
                          schedule_type='polynomial', schedule_rho=7, afs=False, metric='dev', coeff=1.15, model_source='edm', solver='dpmpp',
                          solver_tea='dpmpp', max_order=2, deis_mode='tab', prompt=None, guidance_rate=1.0, predict_x0=True, lower_order_final=True)
                torch.manual_seed(0)
                g0 = time.time()
                dp_list = gits_utils.get_dp_list(net, dev, **gk)
                kw.update(t_steps=solver_utils.get_schedule(61, 0.002, 80, device=dev, dp_list=dp_list), max_order=2, predict_x0=True,
                          lower_order_final=True)
                ent['gits'] = dict(dp_list=[int(v) for v in dp_list], seconds=time.time() - g0, teacher='dpm_pp(2M) on the 61-point polynomial grid, 16 warm-up latents')
            elif a.solver == 'ipndm':
                kw.update(max_order=4)
            elif a.solver == 'dpm_pp':
                kw.update(max_order=2, predict_x0=True)
            ent['build_s'] = time.time() - t0
            sync = torch.cuda.synchronize
            step = lambda: sampler(net, latents, **kw)
            for _ in range(3):
                step()
            clocks = ClockSampler(dev.index or 0)
            clocks.start()
            ms, images = timed_steps(step, args.config_steps, sync, dev, 1)
            ent['clocks'] = clocks.stop()
            if dumps is not None:
                dumps[f'config{c["id"]}_samples'] = images.cpu()
            ent['value'] = a.batch * args.config_steps / (ms / 1e3)
            ent['unit'] = 'images/s (1 GPU)'
            ent['ms_per_step'] = ms / args.config_steps
            ent['e2e'] = measure_e2e(sampler, net, kw, tuple(latents.shape), args.config_steps, sync, dev, 1)
            sub = {}
            roofline_leg(a, sub, net, latents, labels, a.batch, dev, pk, kw)
            ent['roofline'] = sub.get('roofline')
            ent['forward_breakdown_ms'] = sub.get('forward_breakdown_ms')
            del net, images
            torch.cuda.empty_cache()
            if args.gpu_eager and a.net != 'sd15':
                try:
                    ent['gpu_eager'] = gpu_eager_leg(a, dev, native_value=ent['value'], t_steps=kw.get('t_steps'), solver_kw={k: kw[k] for k in ('max_order', 'predict_x0', 'lower_order_final') if k in kw})
                except Exception as e:
                    ent['gpu_eager'] = dict(error=repr(e))
        except Exception as e:
            ent['error'] = repr(e)
        out.append(ent)
        torch.cuda.empty_cache()
    return out


def gpu_eager_leg(args, dev, native_value, t_steps=None, solver_kw=None):
    """The reference's GPU path on this B200: eager PyTorch (cuDNN convolutions, cuBLAS einsum attention, ATen elementwise solver steps)
    through oracle/'s functional restatement of the reference modules (networks_edm.py:60-82 conv2d path, :96-98 group_norm, :105-118
    attention; solvers.py loops), same net / batch / NFE / latents shape.  Three settings:
      default  torch defaults, which is what sample.py runs with: cuDNN TF32 convolutions on, fp32 matmuls (sample.py sets no flags)
      fp32     TF32 off everywhere (the numerics our 1e-3 contract is stated against)
      fp16     the model body in fp16 as EDMPrecond(use_fp16=True) does (networks_edm.py:486) -- the fastest the reference can run
    ratio_* = native images/s / eager images/s on the same GPU in the same process."""
    import torch
    from oracle import edm_oracle as O
    from oracle import solvers_oracle as SO
    P, S = O.make_net(args.net, seed=0, dezero=True)
    P = {k: v.to(dev) for k, v in P.items()}
    B = args.batch
    g = torch.Generator(device=dev).manual_seed(99)
    lat = torch.randn(B, S['img_channels'], S['img_resolution'], S['img_resolution'], generator=g, device=dev)
    lab = None
    if S['label_dim']:
        lab = torch.eye(S['label_dim'], device=dev)[torch.randint(S['label_dim'], (B,), generator=g, device=dev)]
    kw = dict(class_labels=lab, num_steps=args.num_steps, **(solver_kw or {}))
    if t_steps is not None:
        kw['t_steps'] = t_steps
    res = dict(note='eager PyTorch on the same GPU (oracle functional nets = the reference modules, bit-identical on CPU); comparator only',
               batch=B, torch=torch.__version__)
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True                     # sample.py:150 (`torch.backends.cudnn.benchmark = True` in the reference's generators)
    try:
        for name, tf32c, tf32m, dt, timed in (('default', True, False, torch.float32, 2), ('fp16', True, False, torch.float16, 2),
                                              ('fp32', False, False, torch.float32, 1)):
            try:
                torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32c, tf32m
                net = O.OracleNet(P, S, dtype=dt)
                with torch.no_grad():
                    out = SO.sample(net, lat, args.solver, **kw)         # warm-up (cuDNN autotune)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(timed):
                        out = SO.sample(net, lat, args.solver, **kw)
                    e1.record()
                    torch.cuda.synchronize()
                v = B * timed / (e0.elapsed_time(e1) / 1e3)
                res[name] = dict(value=v, unit='images/s (1 GPU)', timed_steps=timed, cudnn_tf32=tf32c, matmul_tf32=tf32m,
                                 dtype=str(dt).replace('torch.', ''), finite=bool(torch.isfinite(out.float()).all()))
                res['ratio_vs_' + name] = native_value / v
                del net, out
            except Exception as e:                   # one setting failing must not hide the others
                res[name] = dict(error=repr(e))
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    return res


def build_sd15(args, dev, B, gen):
    """BASELINE config 5: SD-v1.5-sized eps-net (seeded random weights), CFG 7.5, random [B,77,768] contexts, AMED plug-in on DPM-Solver++(2M),
    num_steps=4 with AFS => NFE=5, 'discrete' schedule rho=1 (amed-solver-main/launch.sh:57)."""
    import math
    import torch
    from diff_sampler_b200 import solvers, solvers_amed
    from diff_sampler_b200.amed_predictor import AMEDPredictor
    from diff_sampler_b200.ldm_net import B200LDMNet
    shapes = sd15_param_shapes()
    g = torch.Generator().manual_seed(777)
    params = {}
    for k, shp in shapes.items():
        if len(shp) == 1:
            v = (torch.rand(shp, generator=g) * 2 - 1) * 0.1
            params[k] = v + 1.0 if k.endswith('.weight') else v
        else:
            fan_in = 1
            for d in shp[1:]:
                fan_in *= d
            params[k] = (torch.rand(shp, generator=g) * 2 - 1) * math.sqrt(3.0 / fan_in)
    net = B200LDMNet(params, img_resolution=64, img_channels=4, num_heads=8, guidance_rate=7.5, precision=args.precision, device=dev)
    c = torch.randn(B, 77, 768, generator=gen, device=dev)
    uc = torch.randn(B, 77, 768, generator=gen, device=dev)
    kw = dict(condition=c, unconditional_condition=uc, num_steps=args.num_steps, sigma_min=net.sigma_min, sigma_max=net.sigma_max,
              schedule_type='discrete', schedule_rho=1)
    if args.solver == 'amed_dpm_pp':
        tg = torch.Generator().manual_seed(4242)
        W = {'map_layer0.weight': torch.randn(8, 8, generator=tg) * 0.3, 'map_layer0.bias': torch.zeros(8),
             'enc_layer0.weight': torch.randn(128, 64, generator=tg) * 0.1, 'enc_layer0.bias': torch.zeros(128),
             'enc_layer1.weight': torch.randn(4, 128, generator=tg) * 0.1, 'enc_layer1.bias': torch.zeros(4),
             'fc_r.weight': torch.randn(1, 20, generator=tg) * 0.2, 'fc_r.bias': torch.zeros(1),
             'fc_scale_time.weight': torch.randn(1, 20, generator=tg) * 0.2, 'fc_scale_time.bias': torch.zeros(1)}
        pred = AMEDPredictor(W, scale_dir=0.0, scale_time=0.2).to(dev)
        kw.update(AMED_predictor=pred, afs=True, max_order=2, predict_x0=False)
        return net, solvers_amed.dpm_pp_sampler, kw
    return net, getattr(solvers, args.solver + '_sampler'), kw


def sd15_param_shapes():
    """UNetModel.state_dict() names/shapes for models/ldm/configs/stable-diffusion/v1-inference.yaml:29-44 (859.5 M parameters)."""
    from collections import OrderedDict
    mc, mult, nrb, attn_res, heads, ctx = 320, (1, 2, 4, 4), 2, (4, 2, 1), 8, 768
    ted = mc * 4
    sh = OrderedDict()

    def lin(n, fi, fo, bias=True):
        sh[n + '.weight'] = (fo, fi)
        if bias:
            sh[n + '.bias'] = (fo,)

    def conv(n, ci, co, k):
        sh[n + '.weight'] = (co, ci, k, k)
        sh[n + '.bias'] = (co,)

    def norm(n, c):
        sh[n + '.weight'] = (c,)
        sh[n + '.bias'] = (c,)

    def res(n, ci, co):
        norm(n + '.in_layers.0', ci); conv(n + '.in_layers.2', ci, co, 3); lin(n + '.emb_layers.1', ted, co)
        norm(n + '.out_layers.0', co); conv(n + '.out_layers.3', co, co, 3)
        if ci != co:
            conv(n + '.skip_connection', ci, co, 1)

    def attn(n, ch):
        t = n + '.transformer_blocks.0'
        norm(n + '.norm', ch); conv(n + '.proj_in', ch, ch, 1)
        for a, cd in (('attn1', ch),):
            lin(f'{t}.{a}.to_q', ch, ch, False); lin(f'{t}.{a}.to_k', cd, ch, False); lin(f'{t}.{a}.to_v', cd, ch, False); lin(f'{t}.{a}.to_out.0', ch, ch)
        lin(f'{t}.ff.net.0.proj', ch, ch * 8); lin(f'{t}.ff.net.2', ch * 4, ch)
        lin(f'{t}.attn2.to_q', ch, ch, False); lin(f'{t}.attn2.to_k', ctx, ch, False); lin(f'{t}.attn2.to_v', ctx, ch, False); lin(f'{t}.attn2.to_out.0', ch, ch)
        for k in (1, 2, 3):
            norm(f'{t}.norm{k}', ch)
        conv(n + '.proj_out', ch, ch, 1)

    lin('time_embed.0', mc, ted); lin('time_embed.2', ted, ted)
    conv('input_blocks.0.0', 4, mc, 3)
    chans, ch, ds, idx = [mc], mc, 1, 1
    for level, m in enumerate(mult):
        for _ in range(nrb):
            res(f'input_blocks.{idx}.0', ch, m * mc); ch = m * mc
            if ds in attn_res:
                attn(f'input_blocks.{idx}.1', ch)
            chans.append(ch); idx += 1
        if level != len(mult) - 1:
            conv(f'input_blocks.{idx}.0.op', ch, ch, 3); chans.append(ch); idx += 1; ds *= 2
    res('middle_block.0', ch, ch); attn('middle_block.1', ch); res('middle_block.2', ch, ch)
    idx = 0
    for level, m in list(enumerate(mult))[::-1]:
        for i in range(nrb + 1):
            res(f'output_blocks.{idx}.0', ch + chans.pop(), mc * m); ch = mc * m
            k = 1
            if ds in attn_res:
                attn(f'output_blocks.{idx}.{k}', ch); k += 1
            if level and i == nrb:
                conv(f'output_blocks.{idx}.{k}.conv', ch, ch, 3); ds //= 2
            idx += 1
    norm('out.0', ch); conv('out.2', mc, 4, 3)
    return sh


# `--precision auto`: the fastest precision whose FINAL IMAGES hold max-abs <= 1e-3 against the reference on that net's BASELINE config
# (de-zeroed random-init weights).  Measured on B200 (profiles/r01d, tests/test_gpu_parity.py::test_fullsize_sampler_parity_f8_mode):
#   cifar10  Heun NFE=18      fp16f8 vs fp16x3 2.7e-4 (+ fp16x3 vs reference <= 1.5e-4)            -> fp16f8
#   imagenet64 DPM++ NFE=10   3.5e-5                                                             -> fp16f8
#   ffhq     iPNDM NFE=6      all blocks in f8: 1.08e-3, over the gate (this net amplifies GEMM rounding the most); f8 only in the blocks
#                             with >= 256 channels (F8_MIN_CHANNELS_FOR): 6.2e-4 at batch 256 (profiles/r02b)     -> fp16f8, f8_min_channels 256
#   sd15     AMED-DPM++ NFE=5  fp16f8 (+ f8_linear) vs fp16x3: 1.4e-2 on latents of magnitude 80 = 1.8e-4 relative (profiles/r02c; the
#                             latent-diffusion tests hold 1e-3 x max|x|, the scale of the random-weight net's latents)      -> fp16f8
PRECISION_FOR = {'cifar10': 'fp16f8', 'imagenet64': 'fp16f8', 'ffhq': 'fp16f8', 'sd15': 'fp16f8'}
# with fp16f8: blocks narrower than this stay fp16x3 (plan.pack_weights).  Only nets whose all-f8 run misses the gate need it.
F8_MIN_CHANNELS_FOR = {'ffhq': 256}


# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of ONE launch of the named GEMM, from `ncu --set full` captures of this
# bench command committed under profiles/ (a number measured under the profiler is a byte count, not a time).
NCU_TRAFFIC = {
    ('conv3x3 256->256 @32x32 x512', 'fp16x3'): (0.539457e9 + 0.496578e9, 'profiles/r01b_ncu_gemm_conv_b512.txt (launch id 1)'),
    ('conv3x3 256->256 @32x32 x512 f8', 'fp16f8'): (0.540013e9 + 0.496059e9, 'profiles/r02/ncu_gemm_pair_cifar_f8_r02p.txt (gemm_tc_pair_kernel, ncu --set full)'),
}


def dominant_launch(args, line, net):
    """Per-launch view of the GEMM shape that takes the largest share of the forward: algorithmic FLOPs and bytes of one launch
    (gemm_desc.describe) over its mean CUDA-event time in this run, plus the ncu DRAM traffic of the same launch where a capture exists."""
    from diff_sampler_b200 import _cstructs as S
    from diff_sampler_b200 import gemm_desc as G
    ms, pl = net.last_profile
    groups = {}
    for i in range(pl.n_ops):
        op = pl.ops_array[i]
        if op.type != S.DS_OP_GEMM:
            continue
        r = G.describe(op.u.gemm)
        g = groups.setdefault(r['label'], dict(n=0, ms=0.0, flops=r['flops'], bytes=r['bytes']))
        g['n'] += 1
        g['ms'] += ms[i]
    label, g = max(groups.items(), key=lambda kv: kv[1]['ms'])
    for (lab, prec), _ in NCU_TRAFFIC.items():            # prefer the shape the committed ncu capture shows, when this plan has it
        if prec == args.precision and lab in groups and groups[lab]['ms'] >= 0.5 * g['ms']:
            label, g = lab, groups[lab]
    per = g['ms'] / g['n']
    traffic = NCU_TRAFFIC.get((label, args.precision))
    rl = line['roofline']
    rl['dominant_launch'] = dict(label=label, launches_per_forward=g['n'], ms_per_launch=per, share_of_gemm_time=g['ms'] / rl['gemm_ms_per_forward'],
                                 algorithmic_flops=g['flops'], achieved_tflops=g['flops'] / (per / 1e3) / 1e12,
                                 frac_of_peak=g['flops'] / (per / 1e3) / 1e12 / rl['peak'], algorithmic_bytes=g['bytes'],
                                 traffic=traffic[0] if traffic else None, traffic_source=traffic[1] if traffic else None)
    if traffic:
        rl['traffic'] = traffic[0]
        rl['traffic_note'] = f'per launch of the dominant GEMM ({label}): algorithmic {g["bytes"] / 1e9:.3f} GB; ' + traffic[1]


def roofline_leg(args, line, net, latents, labels, B, dev, pk, kw):
    """Roofline of the dominant kernel (the tcgen05 GEMM / conv kernel), measured live: every op of one denoiser evaluation is bracketed by
    CUDA events on the launch stream (ds_unet_set_profiling); achieved = algorithmic FLOPs of one evaluation / summed GEMM time."""
    import torch
    from diff_sampler_b200 import _cstructs as S
    x = latents * 2.0
    if hasattr(net, 'profile_call'):                 # latent-diffusion net (CFG: 2B samples per evaluation)
        prof, _ = net.profile_call(x, torch.tensor([2.0], device=dev), kw['condition'], kw['unconditional_condition'])
    else:
        prof = net.profile_forward(x, torch.tensor(2.0, device=dev), labels)
    gemm_n, gemm_ms = prof.get(S.DS_OP_GEMM, (0, 0.0))
    attn_n, attn_ms = prof.get(S.DS_OP_ATTN, (0, 0.0))
    fwd_ms = sum(v[1] for v in prof.values())
    flops = GFLOP_PER_IMG_NFE.get(args.net, 0.0) * 1e9 * B
    tc_ms = gemm_ms + attn_ms                        # all tensor-core kernels: the fused attention kernel carries part of the algorithmic FLOPs
    achieved = flops / (tc_ms / 1e3) / 1e12 if tc_ms > 0 else None
    peak = pk['tflops_sustained']
    # forward time without the per-op events: N evaluations back to back between two events (what a sampler step actually pays per NFE)
    n_rep = 5
    if hasattr(net, 'profile_call'):
        call = lambda: net(x, torch.tensor([2.0], device=dev), condition=kw['condition'], unconditional_condition=kw['unconditional_condition'])
    else:
        call = lambda: net(x, torch.tensor(2.0, device=dev), class_labels=labels)
    call()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(n_rep):
        call()
    f1.record()
    torch.cuda.synchronize()
    line['roofline'] = dict(bound='tensor', achieved=achieved, peak=peak, unit='TFLOP/s', frac=(achieved / peak) if achieved else None,
                            traffic=None, kernel='gemm_tc_pair_kernel / gemm_tc_kernel (+ attn3_kernel): all conv / linear / attention contractions of one denoiser evaluation',
                            algorithmic_flops_per_forward=flops, launches_per_forward=gemm_n + attn_n, gemm_ms_per_forward=gemm_ms,
                            attn_ms_per_forward=attn_ms, all_ops_ms_per_forward=fwd_ms, forward_ms_back_to_back=f0.elapsed_time(f1) / n_rep,
                            gemm_share_of_forward=tc_ms / fwd_ms if fwd_ms else None,
                            executed_mma_flops_factor={'fp16x3': 3, 'fp16f8': 2}.get(args.precision, 1),
                            executed_frac_of_peak=(achieved / peak * {'fp16x3': 3, 'fp16f8': 2}.get(args.precision, 1)) if achieved else None,
                            peak_source=pk['source'] + ', sustained bf16 GEMM',
                            note='frac = algorithmic FLOPs / time / peak; every product costs executed_mma_flops_factor MMA units under the 1e-3 contract '
                                 '(DESIGN.md section 2), so frac <= 1 / factor; executed_frac_of_peak is the tensor-pipe view')
    line['forward_breakdown_ms'] = {OP_NAMES.get(k, str(k)): round(v[1], 4) for k, v in sorted(prof.items())}


OP_NAMES = {1: 'gemm', 2: 'gn_stats', 3: 'gn_apply', 4: 'softmax', 5: 'posemb', 6: 'linear', 7: 'prep_input', 8: 'chanmean', 9: 'memset',
            10: 'layernorm', 11: 'geglu', 12: 'gn_finalize', 13: 'attn'}


def extras(args, line, net, sampler, kw, latents, labels, images, B, dev, pk):
    import torch
    from diff_sampler_b200 import solver_utils
    from diff_sampler_b200.net import B200Net
    from diff_sampler_b200 import _cstructs as S
    if True:
        roofline_leg(args, line, net, latents, labels, B, dev, pk, kw)
        if hasattr(net, 'profile_forward'):
            try:
                dominant_launch(args, line, net)
            except Exception as e:               # diagnostic detail only; the aggregate roofline above stands on its own
                line['roofline']['dominant_launch_error'] = repr(e)
        # ---- the fused solver-update kernel against the HBM roofline (HBM-resident size: 3 x 1 GiB streams) -------------
        n = 256 * 1024 * 1024
        a, b_, c = (torch.empty(n, device=dev).normal_() for _ in range(3))
        a, b_, c = a.view(1024, -1), b_.view(1024, -1), c.view(1024, -1)
        for _ in range(3):
            solver_utils.solver_update(c, a, [1.0, 0.3], mode=S.DS_M_EPS, D=b_, t=2.0)
        torch.cuda.synchronize()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        for _ in range(10):
            solver_update_out = solver_utils.solver_update(c, a, [1.0, 0.3], mode=S.DS_M_EPS, D=b_, t=2.0)
        u1.record()
        torch.cuda.synchronize()
        gbs = 3 * n * 4 * 10 / (u0.elapsed_time(u1) / 1e3) / 1e9
        line['roofline_update'] = dict(bound='hbm', achieved=gbs, peak=pk['hbm_gbs'], unit='GB/s', frac=gbs / pk['hbm_gbs'],
                                       kernel='update_kernel<0, EPS> (Euler step: read x, D; write x+)', bytes_per_launch=3 * n * 4,
                                       peak_source=pk['source'])
        # the same kernel at the BASELINE shape (Heun corrector on [B,3,32,32]: read x, x_pred, D', d; write x+ = 20 B/elem): these
        # 6 MB tensors live in the 126 MB L2, so this is an effective (L2-assisted) bandwidth, reported beside the HBM-resident number
        xs_ = [torch.randn_like(latents) for _ in range(5)]
        for _ in range(5):
            solver_utils.solver_update(xs_[4], xs_[0], [1.0, 0.1, 0.1], mode=S.DS_M_EPS, D=xs_[1], xs=xs_[2], t=2.0, hist=[xs_[3]])
        torch.cuda.synchronize()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        for _ in range(200):
            solver_utils.solver_update(xs_[4], xs_[0], [1.0, 0.1, 0.1], mode=S.DS_M_EPS, D=xs_[1], xs=xs_[2], t=2.0, hist=[xs_[3]])
        v1.record()
        torch.cuda.synchronize()
        us = v0.elapsed_time(v1) / 200 * 1e3
        line['roofline_update']['at_baseline_shape'] = dict(shape=list(latents.shape), bytes_per_launch=5 * latents.numel() * 4, us_per_launch=us,
                                                            effective_gbs=5 * latents.numel() * 4 / (us * 1e-6) / 1e9,
                                                            note='back-to-back launches incl. host launch cadence; tensors are L2-resident')
        del a, b_, c, xs_
        # ---- single-pass fp16 (reported, not the headline: misses the 1e-3 gate on O(1) random nets) -------------------
        if args.precision == 'fp16x3' and args.net != 'sd15':
            net1 = B200Net.from_config(args.net, seed=0, dezero=True, precision='fp16', device=dev)
            for _ in range(2):
                sampler(net1, latents, **kw)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(args.steps):
                img1 = sampler(net1, latents, **kw)
            f1.record()
            torch.cuda.synchronize()
            line['fp16_single_pass'] = dict(value=B * args.steps / (f0.elapsed_time(f1) / 1e3), unit='images/s (1 GPU)',
                                            max_abs_vs_fp16x3=(img1 - images).abs().max().item(),
                                            note='single tcgen05 pass per product; not the headline because it does not hold 1e-3 on the de-zeroed weight set')
            del net1
        # ---- fp16f8 runs: the same sampling pass with the default fp16x3 denoiser, for the speed ratio and the output difference ----
        if args.precision == 'fp16f8':
            import copy
            a3 = copy.copy(args)
            a3.precision, a3.f8_min_channels = 'fp16x3', 0
            net3 = build_workload(a3, dev, int(os.environ.get('RANK', '0')))[0]      # same seeds -> the same weights, latents and contexts
            for _ in range(2):
                sampler(net3, latents, **kw)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(args.steps):
                img3 = sampler(net3, latents, **kw)
            f1.record()
            torch.cuda.synchronize()
            line['fp16x3_same_run'] = dict(value=B * args.steps / (f0.elapsed_time(f1) / 1e3), unit='images/s (1 GPU)',
                                           max_abs_vs_fp16f8=(img3 - images).abs().max().item(), max_abs_image=img3.abs().max().item())
            del net3


if __name__ == '__main__':
    main()
