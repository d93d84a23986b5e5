#!/usr/bin/env python
"""Time the device SSIM (eld_eval_ssim) and what it adds to ELDModel.eval; the float64 CPU oracle for context.
    python tools/eval_bench.py [--calls 400] [--out eval_bench.json]

eld_eval_ssim is timed with CUDA events over --calls calls after a warm-up, at the two shapes the ELD evaluation uses
(one full packed frame, crop=False; a batch of 512^2 centre crops), in two modes:
  l2   back to back: the inputs stay in the 126 MB L2 between calls, as right after eval_apply_kernel wrote them;
  hbm  a 512 MB buffer is written between calls (outside the timed window), so the inputs come from HBM.
Bytes are the 8 B per element the kernel must read (two f32 planes); the floor is bytes / 7.7 TB/s (data-sheet HBM).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {'torch_name': torch.cuda.get_device_name(), 'nvidia_smi': q.stdout.strip() or q.stderr.strip()}


def time_ssim(model, p, t, calls, flush):
    from eld_b200 import _lib
    for _ in range(20):
        model.eval_ssim(p, t)
    torch.cuda.synchronize()
    l0 = _lib.launch_count(0)
    model.eval_ssim(p, t)
    launches = _lib.launch_count(0) - l0
    if flush is None:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            model.eval_ssim(p, t)
        b.record()
        torch.cuda.synchronize()
        per = [a.elapsed_time(b) * 1e3 / calls]
    else:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
        for a, b in ev:
            flush.add_(1.0)
            a.record()
            model.eval_ssim(p, t)
            b.record()
        torch.cuda.synchronize()
        per = [a.elapsed_time(b) * 1e3 for a, b in ev]
    nbytes = 8 * p.numel()
    us = float(np.median(per))
    return {'us_per_call_median': us, 'us_per_call_mean': float(np.mean(per)), 'us_per_call_min': float(np.min(per)),
            'calls': calls, 'bytes': nbytes, 'GB_per_s': nbytes / us / 1e3,
            'hbm_floor_us': nbytes / HBM_BYTES_PER_S * 1e6, 'share_of_hbm_floor': nbytes / HBM_BYTES_PER_S * 1e6 / us,
            'launches_per_call': launches}


def time_eval(model, d, reps, with_ssim):
    """host wall time of ELDModel.eval(correct=True, crop=False), which ends in a device-to-host read"""
    if not with_ssim:
        const = torch.ones(1, device='cuda')
        model.eval_ssim = lambda p, t: const             # the eval of the parent commit: PSNR only
    try:
        for _ in range(3):
            model.eval(d, correct=True, crop=False)
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            model.eval(d, correct=True, crop=False)
            ts.append((time.perf_counter() - t0) * 1e3)
    finally:
        model.__dict__.pop('eval_ssim', None)
    return {'ms_median': float(np.median(ts)), 'ms_min': float(np.min(ts)), 'reps': reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=400)
    ap.add_argument('--eval-reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'eval_bench.py measures the GPU: no device found'
    from eld_b200 import models
    from oracle import eval_ref
    from tests import ssim_ref
    import tempfile
    res = {'card': card(), 'kernel': {}}
    m = models.eld_model()
    m.initialize(models.default_opt(name='eval_bench', checkpoints_dir=tempfile.mkdtemp(), isTrain=False))
    flush = torch.empty(128 * 1024 * 1024, device='cuda')       # 512 MB
    g = torch.Generator(device='cuda').manual_seed(0)
    for name, shape in (('full_frame_1x4x1424x2128', (1, 4, 1424, 2128)), ('crops_8x4x512x512', (8, 4, 512, 512))):
        t = torch.rand(*shape, device='cuda', generator=g)
        p = (t + 0.05 * torch.randn(*shape, device='cuda', generator=g)).contiguous()
        res['kernel'][name] = {'l2': time_ssim(m, p, t, args.calls, None), 'hbm': time_ssim(m, p, t, args.calls, flush)}
        print(name, json.dumps(res['kernel'][name]))
    del flush
    gc = torch.Generator().manual_seed(1)
    t = torch.rand(1, 4, 1424, 2128, generator=gc)
    d = {'input': (t * 0.3 + 0.01 * torch.randn(1, 4, 1424, 2128, generator=gc)).clamp(0, 1), 'target': t, 'fn': ['x']}
    res['eld_model_eval_full_frame'] = {'with_ssim': time_eval(m, d, args.eval_reps, True),
                                        'without_ssim': time_eval(m, d, args.eval_reps, False)}
    print('ELDModel.eval', json.dumps(res['eld_model_eval_full_frame']))
    X, Y = eval_ref.tensor2im(d['input'].numpy()), eval_ref.tensor2im(t.numpy())
    cpu = {}
    for name, (a, b) in (('full_frame_1424x2128x4', (X, Y)), ('crop_512x512x4', (X[:512, :512], Y[:512, :512]))):
        t0 = time.perf_counter()
        ssim_ref.ssim(a, b)
        cpu[name] = {'s_per_frame': time.perf_counter() - t0}
    res['cpu_oracle_float64'] = cpu
    print('CPU oracle', json.dumps(cpu))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
