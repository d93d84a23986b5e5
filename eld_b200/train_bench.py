"""bench.py's U-Net workloads: the training step (BASELINE configs[2]) - noise kernel -> U-Net fwd + L1 + bwd ->
(bucketed NCCL all-reduce overlapped with backward) -> fused Adam - and the inference step (configs[1]), one process
per GPU; plus the ON-BOX baseline: the reference module through PyTorch-eager / cuDNN on the same GPU (SURVEY 2.2)."""
import os
import time

import torch

from . import arch

SONY = (2.2881136684755243, 6.4508722699636545, 15583, 208.9766365993794)
FRAME_BYTES = 4 * 512 * 512 * 8          # algorithmic bytes of the noise kernel per frame (f32 in + f32 out)


def _peaks():
    import bench as _b
    return _b.peaks()


def _tensor_roofline(recs, exclude=('conv10',)):
    """All tcgen05 launches of the recorded step: sum of algorithmic FLOPs / sum of launch times (CUDA events on the
    launch stream), against the BURST cuBLAS bf16 peak: the step runs at ~1.95 GHz and a few hundred watts, not in the
    power-limited regime the sustained figure was measured in (MEASURED_PEAKS.clocks_under_load: 1245 MHz)."""
    tens = [r for r in recs if r['name'].split('.')[1] in ('fprop', 'dgrad', 'wgrad', 'fprop+head') and not r['name'].startswith(exclude)]
    t_ms = sum(r['ms'] for r in tens)
    fl = sum(r['flops'] for r in tens)
    total_ms = sum(r['ms'] for r in recs)
    hbm_peak, tf_peak, tf_sus, _src = _peaks()
    ach = fl / (t_ms * 1e-3) / 1e12
    return {'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': ach / tf_peak,
            'frac_of_sustained_peak': ach / tf_sus, 'traffic': None,
            'kernel': 'conv_umma_kernel + wgrad_conv_kernel (all %d tcgen05 launches of a step)' % len(tens),
            'algorithmic_flops_per_step': fl, 'tensor_ms_per_step': t_ms, 'all_kernels_ms_per_step': total_ms,
            'share_of_step': t_ms / total_ms,
            'peak_kind': 'bf16_tflops (burst cuBLAS peak; kernels run unthrottled at ~1.95 GHz)'}


def onbox_baseline(batch, train, steps=6, warmup=3):
    """The reference's own GPU path on THIS GPU (SURVEY 2.2: 'the on-box bar to beat'): the reference module
    (oracle/unet_ref.py restates models/arch/Unet.py:6-91 line by line) through PyTorch eager -> cuDNN, same batch, same
    step (fwd + L1 + bwd + Adam, ELD_model.py:469-475), U-Net only (the reference makes its noise on the CPU).
    Three precisions: fp32 with TF32 off (what 'fp32' literally is), torch's default (cuDNN may use TF32), and
    bf16 autocast + channels_last (the best cuDNN can do).  frames/s each; baseline only, never on the product path."""
    from oracle import unet_ref
    dev = torch.device('cuda', torch.cuda.current_device())
    out = {}

    def run(tag, tf32, bf16):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.benchmark = True                     # train_syn.py:17
        torch.manual_seed(2018)
        net = unet_ref.UNetSeeInDarkRef(4, 4).to(dev)
        x = torch.rand(batch, 4, 512, 512, device=dev)
        t = torch.rand(batch, 4, 512, 512, device=dev)
        if bf16:
            net = net.to(memory_format=torch.channels_last)
            x, t = x.contiguous(memory_format=torch.channels_last), t.contiguous(memory_format=torch.channels_last)
        opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.999), weight_decay=0) if train else None

        def one():
            with torch.autocast('cuda', dtype=torch.bfloat16, enabled=bf16):
                if train:
                    o = net(x)
                    opt.zero_grad()
                    loss = torch.nn.functional.l1_loss(o.float(), t)
                else:
                    with torch.no_grad():
                        net(x)
                    return
            loss.backward()
            opt.step()
        for _ in range(warmup):
            one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        torch.cuda.synchronize()
        out[tag] = batch * steps / (e0.elapsed_time(e1) * 1e-3)
        del net, opt, x, t
        torch.cuda.empty_cache()
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    try:
        run('fp32_tf32_off_frames_s', False, False)
        run('fp32_torch_default_tf32_conv_frames_s', True, False)
        run('bf16_autocast_channels_last_frames_s', True, True)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b
        torch.backends.cudnn.benchmark = False
    out['what'] = ('reference UNetSeeInDark via PyTorch-eager/cuDNN on this GPU, batch %d x 4x512x512, %s, U-Net only; %d steps after %d warm-ups'
                   % (batch, 'fwd+L1+bwd+Adam' if train else 'forward (no_grad)', steps, warmup))
    return out


def make_train_steps(a, nm, dev, rank, world):
    B = a.batch
    torch.manual_seed(2018)                       # same init on every rank (reference default --seed 2018)
    net = arch.unet(4, 4).to(dev)
    opt = arch.FusedAdam(net, lr=1e-4, betas=(0.9, 0.999), weight_decay=0.0)
    torch.manual_seed(2018 + rank)
    # two alternating clean batches; a step touches ~2.7 GB of activations so nothing survives in L2
    clean = [torch.rand(B, 4, 512, 512, device=dev) for _ in range(2)]
    noisy = torch.empty_like(clean[0])
    loss = torch.zeros((), device=dev)
    plist = [SONY] * B
    host_clean = torch.rand(B, 4, 512, 512).pin_memory()
    host_losses = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_read = [torch.cuda.Event() for _ in range(2)]

    # Optional software pipeline (ELD_OVERLAP=1): the noise kernel of step i+1 on a side stream WHILE step i's network runs
    # (one noise launch per step, all inside the timed region; double-buffered `noisy`, events both ways).  Measured on
    # B200 (profiles/r02_overlap_ab.txt): 4.05 ms overlapped vs 4.00 ms serial - the noise CTAs that do co-reside with
    # the persistent tiles take issue slots from their epilogue warps, which are the tiles' bottleneck on the thin layers.
    # Off by default.
    overlap = os.environ.get('ELD_OVERLAP') is not None
    noise_stream = torch.cuda.Stream(device=dev)
    noisy2 = [noisy, torch.empty_like(noisy)]
    made = [torch.cuda.Event() for _ in range(2)]
    used = [torch.cuda.Event() for _ in range(2)]
    pipe = {'have': None}

    def issue_noise(i, target, after=None):
        k = i & 1
        with torch.cuda.stream(noise_stream):
            noise_stream.wait_event(used[k])                 # the step that last read noisy2[k] has consumed it
            if after is not None:
                noise_stream.wait_event(after)               # e2e: the H2D copy of this clean batch
            nm.batch_gpu(target, params=plist, frame_id0=(i * world + rank) * B, out=noisy2[k])
            made[k].record(noise_stream)
        pipe['have'] = i

    def body(target, i, next_target=None, next_after=None):
        cur = torch.cuda.current_stream()
        k = i & 1
        if overlap:
            if pipe['have'] != i:                            # pipeline start: nothing was made ahead for this step
                here = torch.cuda.Event()
                here.record(cur)
                issue_noise(i, target, here)                 # `target` is ready on the current stream at this point
            cur.wait_event(made[k])
            x = noisy2[k]
        else:
            x = noisy
            nm.batch_gpu(target, params=plist, frame_id0=(i * world + rank) * B, out=noisy)
        if world > 1:
            out, _ = net.train_step_ddp(x, target, loss_out=loss)
        else:
            out, _ = net.train_step(x, target, loss_out=loss)
        if overlap:
            used[k].record(cur)
            if next_target is not None:
                issue_noise(i + 1, next_target, next_after)  # queued behind nothing: runs next to this step's tiles
        opt.step(grad_scale=1.0 / world)
        return {'noisy': x, 'output': out, 'loss': loss, 'weights': net.flat_params}

    def step(i):
        return body(clean[i & 1], i, clean[(i + 1) & 1])

    # end to end: every step's clean batch comes from pinned host memory.  Like a DataLoader with
    # pin_memory + prefetch (train_syn.py:78-80) the copy of batch i+1 runs on a side stream while step i
    # computes; every copy and the D2H of the loss are inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    dev_bufs = [torch.empty(B, 4, 512, 512, device=dev) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {'next': None}

    def issue_copy(i):
        k = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k])            # the step that last read this buffer is done
            dev_bufs[k].copy_(host_clean, non_blocking=True)
            copied[k].record(copy_stream)

    def step_e2e(i):
        k = i & 1
        if state['next'] != i:
            issue_copy(i)
            pipe['have'] = None                            # (re)start of an e2e run: no pre-made input
        cur = torch.cuda.current_stream()
        cur.wait_event(copied[k])
        issue_copy(i + 1)
        state['next'] = i + 1
        body(dev_bufs[k], i, dev_bufs[(i + 1) & 1], copied[(i + 1) & 1])
        consumed[k].record(cur)
        # the loss of EVERY step is read back to the host; the host waits for step i-1's value after it has queued step i
        # (a training loop that logs with one step of lag), so its launch work never leaves the GPU idle.  bench.py's
        # barrier after the timed loop collects the last one.
        host_losses[k].copy_(loss.reshape(1), non_blocking=True)
        loss_read[k].record(cur)
        if state.get('prev') is not None:
            loss_read[state['prev']].synchronize()
        state['prev'] = k

    # ---- live per-launch profile for the roofline entries (a separate, untimed pass) ---------------
    extra = {}
    nm.batch_gpu(clean[0], params=plist, frame_id0=0, out=noisy)
    recs = net.profile(noisy, clean[0], steps=3)
    extra['roofline'] = _tensor_roofline(recs)
    # the noise launch INSIDE the step (between two steps' worth of U-Net traffic: cold L2, like the timed region)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(4)]
    for i, (e0, e1) in enumerate(evs):
        e0.record()
        nm.batch_gpu(clean[i & 1], params=plist, frame_id0=i * B, out=noisy)
        e1.record()
        net.train_step(noisy, clean[i & 1], loss_out=loss)
    torch.cuda.synchronize()
    nms = sorted(e0.elapsed_time(e1) for e0, e1 in evs)[len(evs) // 2]
    hbm_peak = _peaks()[0]
    ach = B * FRAME_BYTES / (nms * 1e-3) / 1e9
    extra['roofline_noise'] = {'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                               'traffic': None, 'kernel': 'noise_packed_*_kernel<%s> (the in-step launch, %d frames)' % (a.model, B),
                               'us_per_launch': nms * 1e3, 'algorithmic_bytes_per_launch': B * FRAME_BYTES,
                               'note': 'exact Poisson is issue-bound, not HBM-bound (DESIGN 5): instructions per pixel, not bytes, set its time'}
    if rank == 0 and world == 1 and not getattr(a, 'no_onbox', False):
        ob = onbox_baseline(B, train=True)
        total_ms = extra['roofline']['all_kernels_ms_per_step']
        ob['ours_unet_step_frames_s'] = B / (total_ms * 1e-3)
        ob['ours_over_best_cudnn'] = ob['ours_unet_step_frames_s'] / max(ob['fp32_tf32_off_frames_s'], ob['fp32_torch_default_tf32_conv_frames_s'],
                                                                          ob['bf16_autocast_channels_last_frames_s'])
        extra['onbox_baseline'] = ob
    return step, step_e2e, host_clean.numel() * 4, 4, extra


def make_infer_steps(a, nm, dev, rank, world):
    """BASELINE configs[1]: U-Net inference on 1 x 4 x 512 x 512 (noisy SonyA7S2 frames).  value: input resident;
    e2e: pinned host frame -> H2D -> forward -> D2H of the restored frame."""
    B = a.batch
    torch.manual_seed(2018)
    net = arch.unet(4, 4).to(dev).eval()
    torch.manual_seed(2018 + rank)
    xs = [nm.batch_gpu(torch.rand(B, 4, 512, 512, device=dev), params=[SONY] * B, frame_id0=k * B) for k in range(4)]
    host_x = xs[0].cpu().pin_memory()

    def step(i):
        return {'output': net(xs[i & 3])}

    # end to end as a three-stage stream pipeline (what a serving loop does): H2D of frame i+1 | forward of frame i | D2H of
    # frame i-1; every frame's input comes from pinned host memory and its restored frame lands in pinned host memory, the
    # host waits for frame i-1 after queueing frame i.
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    dev_xs = [torch.empty_like(xs[0]) for _ in range(2)]
    host_ys = [torch.empty_like(host_x).pin_memory() for _ in range(2)]
    e_in, e_free, e_done, e_out = ([torch.cuda.Event() for _ in range(2)] for _ in range(4))
    st = {'next': None, 'prev': None, 'keep': [None, None]}

    def copy_in(i):
        k = i & 1
        with torch.cuda.stream(s_in):
            s_in.wait_event(e_free[k])
            dev_xs[k].copy_(host_x, non_blocking=True)
            e_in[k].record(s_in)

    def step_e2e(i):
        k = i & 1
        if st['next'] != i:
            copy_in(i)
            st['prev'] = None
        cur = torch.cuda.current_stream()
        cur.wait_event(e_in[k])
        copy_in(i + 1)
        st['next'] = i + 1
        y = net(dev_xs[k])
        e_free[k].record(cur)
        e_done[k].record(cur)
        st['keep'][k] = y                                   # alive until its D2H copy has run
        with torch.cuda.stream(s_out):
            s_out.wait_event(e_done[k])
            host_ys[k].copy_(y, non_blocking=True)
            e_out[k].record(s_out)
        if st['prev'] is not None:
            e_out[st['prev']].synchronize()
        st['prev'] = k

    extra = {}
    recs = net.profile_forward(xs[0], steps=5)
    extra['roofline'] = _tensor_roofline(recs)
    if rank == 0 and world == 1 and not getattr(a, 'no_onbox', False):
        ob = onbox_baseline(B, train=False, steps=20, warmup=5)
        ob['ours_forward_frames_s'] = B / (extra['roofline']['all_kernels_ms_per_step'] * 1e-3)
        extra['onbox_baseline'] = ob
    return step, step_e2e, host_x.numel() * 4, host_ys[0].numel() * 4, extra
