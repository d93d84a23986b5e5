#!/usr/bin/env python
"""bench.py - benchmarks of the ELD synthetic-noise training path on B200 (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload train|infer|noise|fullframe] [--impl reference]
                    [--dump-outputs DIR]

Workloads = BASELINE.json configs (a "frame" is one 4x512x512 packed raw tensor unless stated):
    train      configs[2]  G+P* noise -> U-Net fwd + L1 + bwd -> (all-reduce) -> Adam, batch 8 per GPU, bf16   [default]
    infer      configs[1]  U-Net inference 1 x 4 x 512 x 512
    noise      configs[0]/[3]  the noise kernel alone (--model P+g | p+g | ELD:P+G+B+R+U ..., --batch frames per GPU)
    fullframe  configs[4]  4-camera sweep over 4256 x 2848 full frames (packed 4 x 1424 x 2128), noise synthesis only
Prints ONE JSON line on rank 0.  DESIGN.md section 7 defines value / e2e / roofline / roofline_noise / onbox_baseline /
cpu_baseline.  `--impl reference` times the reference's own CPU path (numpy / torch-CPU port under oracle/) and never
imports the product package.  `--dump-outputs DIR` saves what the last timed step computed as DIR/<name>.npy (rank 0);
the inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

SONY = (2.2881136684755243, 6.4508722699636545, 15583, 208.9766365993794)
FRAME_PX = 4 * 512 * 512
FULL_H, FULL_W = 1424, 2128                      # packed full frame of a 2848 x 4256 sensor (config 5)
METRIC = 'raw frames/sec (noise+U-Net)'
DUMP_SAMPLE = 1 << 22                            # elements kept of a larger output: 16 MB in f32, <= 4 outputs per workload
DUMP_LIMIT = 64 << 20


def peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['hbm_gbs'], d['bf16_tflops'], d.get('bf16_tflops_sustained', d['bf16_tflops']), 'measured'
    return 6650.0, 1590.0, 1400.0, 'fallback'


def ncu_traffic():
    """DRAM bytes per launch from the committed ncu capture of this command (profiles/ncu_traffic.json, written by
    tools/ncu_step_table.py from an `ncu --set full`-metric pass); None if no capture is committed."""
    p = os.path.join(REPO, 'profiles', 'ncu_traffic.json')
    try:
        return json.load(open(p))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  Started BEFORE warm-up and only handed
    back once its first row has arrived, so that nvidia-smi's start-up (it enumerates every GPU of the box) is over
    before the timed window opens - at N = 8 that start-up used to land inside an 80 ms window on rank 0 only."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index, period_ms=25):
        self.index = index
        self.rows = []
        self.proc = None
        self.period_ms = period_ms
        self.t0 = self.t1 = None

    def start(self, wait_s=20.0):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t_end = time.time() + wait_s
            while not self.rows and time.time() < t_end and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def window(self, opening):
        if opening:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 - 0.03 <= t <= (self.t1 or t) + 0.06)]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU legs: the oracle port of the reference path (the only places bench.py executes oracle/).
# Nothing below this line up to main() imports eld_b200.
# ------------------------------------------------------------------------------------------------
def _cpu_noise_frames(args):
    model, nframes, seed, h, w = args
    import numpy as np
    from oracle import ref_numpy
    nm = ref_numpy.NoiseModelRef(model, include=4)
    np.random.seed(seed)
    y = np.random.rand(4, h, w).astype(np.float32)
    t0 = time.perf_counter()
    for _ in range(nframes):
        z = nm(y, params=SONY)
        z = np.maximum(np.minimum(z, 1.0), 0)
    return time.perf_counter() - t0


def _ref_model(model):
    """the reference implements only P / p / g (noise.py:158-166); the paper-restated terms have no reference CPU
    implementation - their CPU leg times the reference's Poisson + Gaussian baseline and says so."""
    return model[4:].replace('G', 'g') if model.startswith('ELD:') else model


def cpu_noise_baseline(model, seconds=12.0, h=512, w=512):
    """Single-thread numpy port of noise.py:149-170 (+clip) on one core, bounded to ~`seconds`."""
    rm = _ref_model(model)
    t1 = _cpu_noise_frames((rm, 1, 2018, h, w))
    n = max(2, int(seconds / t1))
    t = _cpu_noise_frames((rm, n, 2018, h, w))
    return {'value': n / t, 'unit': 'frames/s', 'cores': 1, 'kind': 'port',
            'sample': '%d frames of 4x%dx%d, numpy port of noise.py model %s, 1 thread' % (n, h, w, rm)}


def cpu_infer_fps(steps=3, threads=None):
    import torch
    from oracle import unet_ref
    n = os.cpu_count() or 1
    best = (0.0, 1)
    for th in sorted({min(n, c) for c in ((threads,) if threads else (16, 32, 64))}):
        torch.set_num_threads(th)
        torch.manual_seed(2018)
        net = unet_ref.UNetSeeInDarkRef(4, 4).eval()
        x = torch.rand(1, 4, 512, 512)
        with torch.no_grad():
            net(x)
            t0 = time.perf_counter()
            for _ in range(steps):
                net(x)
        f = steps / (time.perf_counter() - t0)
        if f > best[0]:
            best = (f, th)
    return best


def cpu_baseline(a):
    if a.workload == 'noise':
        return cpu_noise_baseline(a.model)
    if a.workload == 'fullframe':
        return cpu_noise_baseline(a.model, seconds=15.0, h=FULL_H, w=FULL_W)
    if a.workload == 'infer':
        fps, th = cpu_infer_fps()
        return {'value': fps, 'unit': 'frames/s', 'cores': th, 'kind': 'port',
                'sample': 'reference module (oracle/unet_ref.py) torch CPU fp32 forward, 1x4x512x512 x 3, %d threads (best of 16/32/64)' % th}
    from oracle import unet_ref
    nb = cpu_noise_baseline(a.model, seconds=6.0)
    fps_unet, nthr = unet_ref.cpu_train_fps_best(steps=2, warmup=1, batch=1)
    fps = 1.0 / (1.0 / nb['value'] + 1.0 / fps_unet)
    return {'value': fps, 'unit': 'frames/s', 'cores': nthr, 'kind': 'port',
            'sample': nb['sample'] + '; U-Net torch CPU fp32 fwd+L1+bwd+Adam, batch 1 x 2 steps, %d threads - best of 16/32/64 (noise leg 1 thread)' % nthr}


def config_dict(a):
    w = a.workload
    if w == 'noise':
        return {'workload': 'noise.py %s sampler, batch %d x 4x512x512 packed raw (SonyA7S2 params), f32 in/out' % (a.model, a.batch),
                'frames_per_step_per_gpu': a.batch, 'cache': 'inputs+outputs %d MiB per step > 126 MiB L2' % (a.batch * 8)}
    if w == 'fullframe':
        return {'workload': '4-camera parameter sweep (include 1..4), %s noise synthesis on 4256x2848 full frames = packed 4x%dx%d f32, '
                            '%d frames per GPU per step, cameras round-robin (BASELINE configs[4])' % (a.model, FULL_H, FULL_W, a.batch),
                'frames_per_step_per_gpu': a.batch, 'cache': 'inputs+outputs %d MiB per step > 126 MiB L2' % (a.batch * 93),
                'equiv_512_frames_per_full_frame': FULL_H * FULL_W / (512.0 * 512.0)}
    if w == 'infer':
        return {'workload': 'U-Net inference 1x4x512x512 (BASELINE configs[1]); bf16 tcgen05 tiles with fp32 accumulation serve the '
                            'fp32 request at rel-L2 <= 2e-2 (DESIGN 5.2)', 'global_batch': a.batch * a.gpus,
                'frames_per_step_per_gpu': a.batch, 'parallelism': 'dp%d' % a.gpus,
                'cache': 'activations of one forward ~180 MB > 126 MiB L2; 4 rotating inputs'}
    return {'workload': 'train_syn.py step: %s noise + U-Net fwd+L1+bwd+Adam, batch %d x 4x512x512 bf16, L1 loss (BASELINE configs[2])' % (a.model, a.batch),
            'global_batch': a.batch * a.gpus, 'frames_per_step_per_gpu': a.batch, 'parallelism': 'dp%d' % a.gpus,
            'cache': 'activations %s > 126 MiB L2' % 'of a step'}


def reference_arm(a):
    """--impl reference: the reference's own CPU implementation of the path (the Python reference cannot be compiled or
    shipped; the numpy/torch oracle port restates it line by line) on all host cores.  One step = the workload's batch
    on the CPU: noise in a multiprocessing pool mirroring DataLoader(num_workers) (train_syn.py:78-80), U-Net
    fwd+L1+bwd+Adam with torch CPU.  The legs run back to back (the reference's DataLoader would overlap them; the
    U-Net leg dominates by > 10x, so the serial sum is within 10 % of the overlapped figure)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    nproc = os.cpu_count() or 1
    w, model = a.workload, _ref_model(a.model)
    h, wd = (FULL_H, FULL_W) if w == 'fullframe' else (512, 512)
    out = {'impl': 'reference', 'metric': METRIC, 'unit': 'frames/s', 'n_gpus': a.gpus,
           'steps': a.steps, 'warmup': a.warmup, 'higher_is_better': True, 'scaling': 'weak',
           'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config_dict(a)}
    noise_fps = None
    if w != 'infer':
        per_step = min(nproc, 16) if w == 'fullframe' else nproc            # one frame per worker per step
        t_noise = []
        with mp.Pool(per_step) as pool:
            for s in range(a.warmup + a.steps):
                t0 = time.perf_counter()
                pool.map(_cpu_noise_frames, [(model, 1, 1000 + s * nproc + i, h, wd) for i in range(per_step)])
                dt = time.perf_counter() - t0
                if s >= a.warmup:
                    t_noise.append(dt)
        noise_fps = per_step * len(t_noise) / sum(t_noise)
    if w in ('noise', 'fullframe'):
        fps = noise_fps
        sample = '%d frames/step of 4x%dx%d in a %d-process pool, numpy port of noise.py model %s' % (per_step, h, wd, per_step, model)
    elif w == 'infer':
        fps, nthr = cpu_infer_fps(steps=a.steps)
        sample = ('reference module torch CPU fp32 forward 1x4x512x512 x %d steps on %d threads (best of 16/32/64; nproc = %d)'
                  % (a.steps, nthr, nproc))
    else:
        from oracle import unet_ref
        fps_unet, nthr = unet_ref.cpu_train_fps_best(steps=a.steps, warmup=1, batch=1)
        fps = 1.0 / (1.0 / noise_fps + 1.0 / fps_unet)
        sample = ('noise: %d frames/step in a %d-process pool (%.1f frames/s); U-Net: torch CPU fp32 fwd+L1+bwd+Adam batch 1 x %d '
                  'steps on %d threads (%.2f frames/s; best of min(nproc, 16/32/64); nproc = %d); legs summed serially'
                  % (per_step, nproc, noise_fps, a.steps, nthr, fps_unet, nproc))
    out.update({'value': fps, 'ms_per_step': 1000.0 * a.batch / fps,
                'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': nproc, 'kind': 'port', 'sample': sample},
                'e2e': {'value': fps, 'unit': 'frames/s', 'steps': a.steps, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0})
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------
def dump_outputs(d, outs):
    """outs: {name: tensor} of one step -> d/<name>.npy, float32 (float64 kept), in the output's shape.  An output of
    n > DUMP_SAMPLE elements is saved flat as exactly DUMP_SAMPLE of its elements: element j is the flat element
    j * n // DUMP_SAMPLE + floor(u_j * size of that range), u = RandomState(0).random_sample(DUMP_SAMPLE), so the sample
    spreads evenly over the output and depends only on n."""
    import numpy as np
    import torch
    os.makedirs(d, exist_ok=True)
    total = 0
    for name, t in sorted(outs.items()):
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            edges = np.arange(DUMP_SAMPLE + 1) * t.numel() // DUMP_SAMPLE
            idx = edges[:-1] + (np.random.RandomState(0).random_sample(DUMP_SAMPLE) * np.diff(edges)).astype(np.int64)
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        arr = t.cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)
        total += arr.nbytes
        assert total <= DUMP_LIMIT, 'outputs exceed %d bytes' % DUMP_LIMIT
        np.save(os.path.join(d, name + '.npy'), arr)


def make_noise_steps(a, dev, rank, world, full):
    import numpy as np
    import torch
    from eld_b200.noise import NoiseModel
    B = a.batch
    h, w = (FULL_H, FULL_W) if full else (512, 512)
    is_full_model = a.model.startswith('ELD:')
    if full:
        # config 5: one NoiseModel per camera (include 1..4), frame i of a step uses camera i % 4's sampled parameters
        nms = [NoiseModel(a.model, include=c, verbose=False, seed=2018) for c in (1, 2, 3, 4)]
        plist = [nms[i % 4].frame_params(1000 + i, 1)[0] for i in range(B)]
        nm = nms[0]
    else:
        nm = NoiseModel(a.model, include=4, verbose=False, seed=2018)
        plist = nm.frame_params(0, B) if is_full_model else [SONY] * B
    torch.manual_seed(2018 + rank)
    # two alternating input/output sets so no step re-reads lines the previous one left in L2
    clean = [torch.rand(B, 4, h, w, device=dev) for _ in range(2)]
    noisy = [torch.empty_like(clean[0]) for _ in range(2)]
    host_in = torch.rand(B, 4, h, w).pin_memory()
    host_out = torch.empty(B, 4, h, w).pin_memory()
    dev_in = torch.empty(B, 4, h, w, device=dev)
    dev_out = torch.empty_like(dev_in)

    def step(i):
        return {'noisy': nm.batch_gpu(clean[i & 1], params=plist, frame_id0=(i * world + rank) * B, out=noisy[i & 1])}

    def step_e2e(i):
        dev_in.copy_(host_in, non_blocking=True)
        nm.batch_gpu(dev_in, params=plist, frame_id0=(i * world + rank) * B, out=dev_out)
        host_out.copy_(dev_out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    return step, step_e2e, host_in.numel() * 4, host_out.numel() * 4, B * 4 * h * w * 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--workload', default='train', choices=['train', 'infer', 'noise', 'fullframe'])
    ap.add_argument('--model', default='P+g', help="noise model string (reference semantics); G+P* = 'P+g'; "
                                                   "'ELD:P+G+B+R+U' = the paper-restated full model")
    ap.add_argument('--batch', type=int, default=None, help='frames per GPU per step')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-onbox', action='store_true', help='skip the torch-eager/cuDNN on-box baseline')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed as DIR/<name>.npy')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.batch is None:
        a.batch = {'train': 8, 'infer': 1, 'noise': 32, 'fullframe': 4}[a.workload]
    a.warmup = max(a.warmup, 3)

    if a.impl == 'reference':
        if a.dump_outputs:
            ap.error('--dump-outputs saves the product path; --impl reference has none')
        return reference_arm(a)

    import torch
    import torch.distributed as dist
    from eld_b200 import _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    assert world == a.gpus, 'launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)' % (a.gpus, world)

    hbm_peak, tf_peak, tf_sus, peak_src = peaks()
    B = a.batch

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None      # one nvidia-smi poller per job, not per rank
    if sampler is not None:
        sampler.start()                                        # before warm-up; returns after its first row
    extra = {}
    if a.workload in ('noise', 'fullframe'):
        step, step_e2e, h2d, d2h, kernel_bytes = make_noise_steps(a, dev, rank, world, a.workload == 'fullframe')
        dtype = 'f32'
    else:
        from eld_b200.noise import NoiseModel
        from eld_b200.train_bench import make_train_steps, make_infer_steps
        nm = NoiseModel(a.model, include=4, verbose=False, seed=2018)
        mk = make_train_steps if a.workload == 'train' else make_infer_steps
        step, step_e2e, h2d, d2h, extra = mk(a, nm, dev, rank, world)
        kernel_bytes = None
        dtype = 'bf16'

    for i in range(a.warmup):
        step(i)
    barrier()
    l0 = _lib.launch_count(local)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    if sampler is not None:
        sampler.window(True)
    ev[0].record()
    for i in range(a.steps - 1):
        step(a.warmup + i)
    last = step(a.warmup + a.steps - 1)             # only the last step's outputs outlive it, for --dump-outputs
    ev[1].record()
    import ctypes
    probe = torch.zeros(1, device=dev)
    _lib.check(_lib.load().eld_clock_probe(_lib.ctx(local), probe.data_ptr(),
                                           ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), 'eld_clock_probe')
    barrier()
    if sampler is not None:
        sampler.window(False)
    clocks = sampler.stop() if sampler is not None else None
    if clocks is not None:
        # the SM clock right behind the last timed kernel, from %clock64 / %globaltimer on the device (nvidia-smi's
        # 25 ms samples cannot resolve an 80 ms window)
        clocks['sm_mhz_device_probe'] = float(probe.item())
    ms = ev[0].elapsed_time(ev[1])
    launches = _lib.launch_count(local) - l0
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, last)              # before the end-to-end steps below move the weights on
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    frames = B * world * a.steps
    value = frames / (ms * 1e-3)

    # end to end through the public API with HOST buffers (pinned), copies inside the timed region
    for i in range(2):
        step_e2e(i)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(3, a.steps // 2)
    for i in range(e2e_steps):
        step_e2e(i)
    barrier()
    te = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = B * world * e2e_steps / float(te.item())

    traffic = ncu_traffic()
    if a.workload in ('noise', 'fullframe'):
        ach = kernel_bytes * a.steps / (ms * 1e-3) / 1e9   # the step IS the kernel
        key = 'noise:%s:%s' % (a.workload, a.model)
        roof = {'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                'traffic': (traffic or {}).get(key), 'kernel': 'noise_packed_*_kernel<%s>' % a.model, 'peak_source': peak_src,
                'algorithmic_bytes_per_launch': kernel_bytes, 'peak_kind': 'hbm_gbs (measured copy bandwidth)'}
    else:
        roof = extra.pop('roofline')
        roof['peak_source'] = peak_src
        if traffic and a.workload in traffic:
            roof['traffic'] = traffic[a.workload].get('tensor_tile_bytes_per_step')
            if 'roofline_noise' in extra:
                extra['roofline_noise']['traffic'] = traffic[a.workload].get('noise_bytes_per_launch')

    out = {'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world,
           'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': ms / a.steps, 'higher_is_better': True,
           'scaling': 'weak', 'vs_baseline': None, 'dtype': dtype, 'data': 'synthetic',
           'config': config_dict(a), 'clocks': clocks,
           'e2e': {'value': e2e_value, 'unit': 'frames/s', 'steps': e2e_steps, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
           'gpu_launches': launches, 'roofline': roof}
    if a.workload == 'fullframe':
        out['equiv_512_frames_per_s'] = value * FULL_H * FULL_W / (512.0 * 512.0)
    out.update(extra)
    if rank == 0:
        if not a.no_cpu_baseline and world == 1:      # the CPU baseline is timed at N = 1 only (the other ranks would idle)
            out['cpu_baseline'] = cpu_baseline(a)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
