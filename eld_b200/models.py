"""Drop-in for the reference's model factory seam (SURVEY 8b): `models.__dict__[opt.model]()`
-> object with initialize / set_input / optimize_parameters / get_current_errors / save / load ...
Reference: models/ELD_model.py:172-200 (set_input), :352-523 (ELDModel), models/base_model.py.

Differences that are the point of this repo
  * netG is eld_b200.arch.unet (tcgen05 engine); forward+L1+backward is ONE C-ABI call, Adam another;
  * noise can be synthesised ON THE TRAINING STREAM (opt.noise_on_gpu / a batch without 'input'):
    only the clean frame crosses PCIe, the fused CUDA kernel makes the noisy input (SURVEY F4);
  * data parallel: if torch.distributed is initialised the flat gradient buffer is all-reduced
    (NCCL over NVLink) between backward and Adam - one collective, U-Net weights only;
  * get_current_errors() keeps the reference's `.item()` host sync but can be told to defer it.
"""
import os
from collections import OrderedDict
from types import SimpleNamespace

import numpy as np
import torch
import torch.distributed as dist

from . import arch


def default_opt(**kw):
    """The flags the hot path reads (reference options/eld/{base,train}_options.py), with defaults."""
    o = dict(name='eld_b200', gpu_ids=[0], model='eld_model', checkpoints_dir='./checkpoints', resume=False,
             resume_epoch=None, seed=2018, chop=False, no_log=True, no_verbose=True, netG='unet', channels=4,
             stage_in='raw', stage_out='raw', model_path=None, include=4, crf=False, batchSize=1, lr=1e-4,
             beta1=0.9, wd=0.0, loss='l1', noise='g', isTrain=True, save_epoch_freq=100, noise_on_gpu=False,
             augment_on_gpu=False, defer_loss_sync=False, prefetch_noise=False, num_burst=1)
    o.update(kw)
    return SimpleNamespace(**o)


class BaseModel:
    """models/base_model.py:6-74"""

    def name(self):
        return self.__class__.__name__.lower()

    def initialize(self, opt):
        self.opt = opt
        self.gpu_ids = opt.gpu_ids
        self.isTrain = opt.isTrain
        self.save_dir = os.path.join(opt.checkpoints_dir, opt.name)
        self._count = 0

    def update_learning_rate(self):
        for scheduler in self.schedulers:
            scheduler.step()
        lr = self.optimizers[0].param_groups[0]['lr']
        print('learning rate = %.7f' % lr)

    def print_optimizer_param(self):
        print(self.optimizers[-1])

    def save(self, label=None):
        # one writer per job: under torch.distributed every replica holds the same state (rank 0 writes, all wait)
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            if dist.get_rank() == 0:
                self._save(label)
            dist.barrier()
            return
        self._save(label)

    def _save(self, label=None):
        epoch, iterations = self.epoch, self.iterations
        if label is None:
            model_name = os.path.join(self.save_dir, 'model' + '_%03d_%08d.pt' % (epoch, iterations))
        else:
            model_name = os.path.join(self.save_dir, 'model' + '_' + label + '.pt')
        os.makedirs(self.save_dir, exist_ok=True)
        torch.save(self.state_dict(), model_name)

    def _init_optimizer(self, optimizers):
        self.optimizers = optimizers
        self.schedulers = []
        for optimizer in self.optimizers:
            for group in optimizer.param_groups:             # util.set_opt_param
                group['initial_lr'] = self.opt.lr
                group['weight_decay'] = self.opt.wd


class ELDModel(BaseModel):
    def __init__(self):
        self.epoch = 0
        self.iterations = 0
        self.device = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else None
        self.noise_maker = None
        self.loss_pixel = None
        self._frames_seen = 0
        self.CRF = None
        self._prefetched = None
        self._noise_stream = None

    def _eval(self):
        self.netG.eval()

    def _train(self):
        self.netG.train()

    def initialize(self, opt, noise_maker=None):
        BaseModel.initialize(self, opt)
        if self.device is None:
            raise RuntimeError('ELDModel (eld_b200) needs a CUDA device: no CPU fallback')
        if len(opt.gpu_ids) > 0:
            self.device = torch.device('cuda', opt.gpu_ids[0])
        if getattr(opt, 'crf', False) and getattr(self, 'CRF', None) is None:
            from . import process
            self.CRF = process.load_CRF()                                                   # ELD_model.py:374-375
        chan = {'raw': opt.channels, 'srgb': 3}                                             # ELD_model.py:377-389
        if opt.stage_in not in chan:
            raise NotImplementedError('Invalid Input Stage: {}'.format(opt.stage_in))
        if opt.stage_out not in chan:
            raise NotImplementedError('Invalid Output Stage: {}'.format(opt.stage_out))
        self.netG = arch.__dict__[opt.netG](chan[opt.stage_in], chan[opt.stage_out]).to(self.device)     # ELD_model.py:391
        self.noise_maker = noise_maker
        if self.isTrain:
            if opt.loss not in ('l1', 'l2'):
                raise NotImplementedError("pixel losses of models/losses.py:29-36: 'l1' (nn.L1Loss) or 'l2' (nn.MSELoss)")
            self.netG.loss_kind = opt.loss
            self.optimizer_G = arch.FusedAdam(self.netG, lr=opt.lr, betas=(opt.beta1, 0.999), weight_decay=opt.wd)
            self._init_optimizer([self.optimizer_G])
        if opt.resume:
            self.load(self, opt.resume_epoch)
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank() if self.world > 1 else 0
        self._sync_replicas()

    def _sync_replicas(self):
        """Data-parallel replicas start from rank 0's weights and Adam moments whatever each rank's torch seed was
        (the reference is single-GPU; train_syn.py seeds every process alike, an Engine caller may not)."""
        if self.world > 1:
            dist.broadcast(self.netG.flat_params, 0)
            if self.isTrain:
                dist.broadcast(self.optimizer_G.m, 0)
                dist.broadcast(self.optimizer_G.v, 0)

    # ---- ELDModelBase.set_input (ELD_model.py:173-200) -------------------------------------------------
    def set_input(self, data, mode='train'):
        mode = mode.lower()
        target, data_name = None, None
        if mode == 'train':
            input, target = data.get('input'), data['target']
        elif mode == 'eval':
            input, target, data_name = data['input'], data['target'], data['fn']
        elif mode == 'test':
            input, data_name = data['input'], data['fn']
        else:
            raise NotImplementedError('Mode [%s] is not implemented' % mode)
        synth = mode == 'train' and (input is None or getattr(self.opt, 'noise_on_gpu', False))
        pre = self._prefetched if synth else None
        if target is not None and not (pre is not None and pre[0] is data):
            target = target.to(device=self.device, dtype=torch.float32, non_blocking=True)
        if synth:
            self._prefetched = None
            if pre is not None and pre[0] is data:
                # made ahead by prefetch_input() on the side stream while the previous step's network ran
                _, input, target, ev = pre
                cur = torch.cuda.current_stream()
                cur.wait_event(ev)
                input.record_stream(cur)
                target.record_stream(cur)
            else:
                input, target = self._synthesize(target)
            if self.opt.stage_in == 'srgb' and input.shape[1] == 4:
                # ISPDataset.__getitem__ (sid_dataset.py:306-312) on the stream: noise -> clip -> raw2rgb_v2(wb, ccm) -> clip
                from . import process
                assert 'wb' in data and 'ccm' in data, "--stage_in srgb needs the frames' (wb, ccm) meta in the batch"
                input = process.isp_dataset_item(input, data['wb'], data['ccm'], CRF=getattr(self, 'CRF', None))
        else:
            input = input.to(device=self.device, dtype=torch.float32, non_blocking=True)
        self.input, self.target, self.data_name = input, target, data_name
        self.rawpath = data['rawpath'][0] if 'rawpath' in data else None
        self.cfa = data['cfa'][0] if 'cfa' in data else 'bayer'
        self.aligned = False if 'unaligned' in data else True

    def _synthesize(self, target):
        """On-the-fly synthesis (SynDataset semantics, sid_dataset.py:259-280, incl. the [0,1] clip) on the CURRENT stream.
        Frame ids count GLOBAL frames: step s of a W-GPU job owns ids [F, F + sum of the ranks' batch sizes), rank r the
        r-th slice.  Batches are equal-sized except possibly the last one of an epoch (DataLoader without drop_last), so F
        advances by the batch actually seen times W - ids never repeat, and the running count is part of the checkpoint
        (a resumed run does not replay the Philox streams from frame 0)."""
        assert self.noise_maker is not None, 'noise_on_gpu needs a noise_maker (eld_b200.noise.NoiseModel)'
        n = target.shape[0]
        fid0 = self._frames_seen + self.rank * n
        self._frames_seen += self.world * n
        # per-frame (K, g_scale, ratio, ...) and flip flags are drawn from a generator keyed by (seed, global frame id):
        # W ranks draw W*n DIFFERENT tuples (not W copies of the same n), and frame f gets the same tuple at any GPU
        # count.  The draw itself is noise.py:201-225's call order on that per-frame RandomState.
        params = self.noise_maker.frame_params(fid0, n, burst=max(1, int(getattr(self.opt, 'num_burst', 1))))
        if getattr(self.opt, 'augment_on_gpu', False):
            # ELDTrainDataset's flips / transpose / clip (sid_dataset.py:340-356) fused into the noise kernel:
            # both the synthesised input and the target come back augmented, one pass over the frames
            return self.noise_maker.batch_gpu_augmented(target, aug=self.noise_maker.frame_augment(fid0, n),
                                                        params=params, frame_id0=fid0, clip=True)
        return self.noise_maker.batch_gpu(target, params=params, frame_id0=fid0, clip=True), target

    def prefetch_input(self, data):
        """Start synthesising the NEXT step's noisy input on a side stream (Engine.train calls this right after it has
        queued the current step): the exact-Poisson noise kernel is issue-bound, the U-Net tiles are tensor / memory
        bound, so the two overlap almost for free.  set_input(data) with the SAME dict then only waits for an event.
        A no-op unless the model synthesises its input (opt.noise_on_gpu or a batch without 'input')."""
        if not (self.isTrain and (data.get('input') is None or getattr(self.opt, 'noise_on_gpu', False))):
            return
        if self._noise_stream is None:
            self._noise_stream = torch.cuda.Stream(device=self.device)
        self._noise_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._noise_stream):
            target = data['target'].to(device=self.device, dtype=torch.float32, non_blocking=True)
            input, target = self._synthesize(target)
            ev = torch.cuda.Event()
            ev.record(self._noise_stream)
        self._prefetched = (data, input, target, ev)

    # ---- forward / optimise (ELD_model.py:411-475) -------------------------------------------------------
    def forward(self):
        if self.opt.chop:
            output = self.forward_chop(self.input)
        else:
            output = self.netG(self.input)
        self.output = output
        return output

    def forward_chop(self, x, base=16):
        """ELD_model.py:434-467: 4 overlapping quadrants; each quadrant is padded up to the tile grid the
        engine needs (H%128, W%256) by replication and cropped back."""
        b, c, h, w = x.size()
        h_half, w_half = h // 2, w // 2
        shave_h = np.ceil(h_half / base) * base - h_half
        shave_w = np.ceil(w_half / base) * base - w_half
        shave_h = shave_h if shave_h >= 10 else shave_h + base
        shave_w = shave_w if shave_w >= 10 else shave_w + base
        h_size, w_size = int(h_half + shave_h), int(w_half + shave_w)
        inputs = [x[:, :, 0:h_size, 0:w_size], x[:, :, 0:h_size, (w - w_size):w],
                  x[:, :, (h - h_size):h, 0:w_size], x[:, :, (h - h_size):h, (w - w_size):w]]
        outputs = [self._padded_forward(i) for i in inputs]
        output = x.new_empty(b, outputs[0].shape[1], h, w)
        output[:, :, 0:h_half, 0:w_half] = outputs[0][:, :, 0:h_half, 0:w_half]
        output[:, :, 0:h_half, w_half:w] = outputs[1][:, :, 0:h_half, (w_size - w + w_half):w_size]
        output[:, :, h_half:h, 0:w_half] = outputs[2][:, :, (h_size - h + h_half):h_size, 0:w_half]
        output[:, :, h_half:h, w_half:w] = outputs[3][:, :, (h_size - h + h_half):h_size, (w_size - w + w_half):w_size]
        return output

    def _padded_forward(self, x):
        """the engine runs any H, W that are multiples of 16 exactly (like the reference network); other sizes
        are replicate-padded up to the next multiple of 16 and cropped (the reference cannot run them at all)."""
        h, w = x.shape[2:]
        H, W = -(-h // 16) * 16, -(-w // 16) * 16
        if (H, W) != (h, w):
            x = torch.nn.functional.pad(x, (0, W - w, 0, H - h), mode='replicate')
        return self.netG(x.contiguous())[:, :, :h, :w]

    def optimize_parameters(self):
        """forward, zero_grad, L1 backward, (all-reduce), Adam - ELD_model.py:469-475."""
        self._train()
        if self.world > 1:
            self.output, self.loss_pixel = self.netG.train_step_ddp(self.input, self.target)
        else:
            self.output, self.loss_pixel = self.netG.train_step(self.input, self.target)
        self.optimizer_G.step(grad_scale=1.0 / self.world)

    def backward_G(self):
        """ELD_model.py:411-420 as written in the reference: loss on self.output, .backward() through the netG autograd
        node.  optimize_parameters() does not use it (the fused step is one C-ABI call) - it exists so that code written
        against the reference's forward() / backward_G() pair keeps working, with any torch loss."""
        loss_fn = torch.nn.functional.l1_loss if self.opt.loss == 'l1' else torch.nn.functional.mse_loss
        self.loss_G = self.loss_pixel = loss_fn(self.output, self.target)
        self.loss_G.backward()

    def get_current_errors(self):
        ret_errors = OrderedDict()
        if self.loss_pixel is not None:
            ret_errors['Pixel'] = self.loss_pixel if getattr(self.opt, 'defer_loss_sync', False) else self.loss_pixel.item()
        return ret_errors

    def eval_metrics(self, predict, target, correct=False):
        """IlluminanceCorrect (ELD_model.py:138-169) + tensor2im (:23-38) + PSNR (util/index.py:76-79) per frame, on the
        device (csrc/eval.cu, three launches, no host synchronisation).  Returns (output, psnr[n], gain[n]) - output is
        the corrected prediction when correct=True, else `predict` itself."""
        import ctypes
        from . import _lib
        predict, target = predict.contiguous(), target.contiguous()
        n = predict.shape[0]
        if target.shape[0] == 1 and n != 1:
            target = target.expand_as(predict).contiguous()     # IlluminanceCorrect.forward's broadcast case (:147-149)
        out = torch.empty_like(predict) if correct else predict
        scratch = torch.empty(n * 4, dtype=torch.float64, device=predict.device)
        psnr = torch.empty(n, dtype=torch.float32, device=predict.device)
        gain = torch.empty(n, dtype=torch.float32, device=predict.device)
        _lib.check(_lib.load().eld_eval_correct_psnr(
            _lib.ctx(predict.device.index or 0), predict.data_ptr(), target.data_ptr(), out.data_ptr() if correct else None, n,
            predict[0].numel(), int(bool(correct)), scratch.data_ptr(), psnr.data_ptr(), gain.data_ptr(),
            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), 'eld_eval_correct_psnr')
        return out, psnr, gain

    def eval_ssim(self, predict, target):
        """tensor2im (ELD_model.py:23-38) + skimage's structural_similarity(data_range=255, multichannel=True) with its
        defaults (util/index.py:80) per frame of NCHW fp32 tensors, on the device (csrc/eval.cu, two launches, no host
        synchronisation).  A 1-frame target is broadcast over the batch like eval_metrics.  Returns ssim[n] (f32)."""
        import ctypes
        from . import _lib
        predict, target = predict.contiguous(), target.contiguous()
        n, c, h, w = predict.shape
        if target.shape[0] == 1 and n != 1:
            target = target.expand_as(predict).contiguous()
        scratch = torch.empty(n * c, dtype=torch.float64, device=predict.device)
        ssim = torch.empty(n, dtype=torch.float32, device=predict.device)
        _lib.check(_lib.load().eld_eval_ssim(
            _lib.ctx(predict.device.index or 0), predict.data_ptr(), target.data_ptr(), n, c, h, w, scratch.data_ptr(),
            ssim.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), 'eld_eval_ssim')
        return ssim

    def illuminance_correct(self, predict, source):
        return self.eval_metrics(predict, source, correct=True)[0]

    def eval(self, data, savedir=None, suffix=None, correct=False, crop=True, frame_id=None, **kwargs):
        """ELDModelBase.eval (ELD_model.py:203-243) without the rawpy / PIL visualisation: centre 512x512 crop
        (util.crop_center), forward (or forward_chop), optional illuminance correction, PSNR and SSIM of the output and
        of the input against the target exactly as tensor2im + quality_assess compute them - all on the device
        (csrc/eval.cu); one host read of the final scalars.  Only the 1st frame is assessed, like the reference
        (tensor2im takes [0])."""
        self._eval()
        self.set_input(data, 'eval')
        with torch.no_grad():
            x, t = self.input, self.target
            if crop and x.shape[2] >= 512 and x.shape[3] >= 512:
                h, w = x.shape[2:]
                y0, x0 = h // 2 - 256, w // 2 - 256                     # util.crop_center
                x, t = x[:, :, y0:y0 + 512, x0:x0 + 512].contiguous(), t[:, :, y0:y0 + 512, x0:x0 + 512].contiguous()
            out = self.forward_chop(x) if self.opt.chop else self._padded_forward(x)
            out, psnr, _ = self.eval_metrics(out.contiguous(), t, correct=correct)
            _, psnr_in, _ = self.eval_metrics(x, t, correct=False)
            ssim = self.eval_ssim(out[:1], t[:1])
            ssim_in = self.eval_ssim(x[:1], t[:1])
            self.output = out
            r = torch.stack([psnr[0], psnr_in[0], ssim[0], ssim_in[0]]).cpu()
        return {'PSNR': float(r[0]), 'PSNR_input': float(r[1]), 'SSIM': float(r[2]), 'SSIM_input': float(r[3])}

    def test(self, data, savedir=None, **kwargs):
        self._eval()
        self.set_input(data, 'test')
        with torch.no_grad():
            return self._padded_forward(self.input)

    # ---- checkpoints (ELD_model.py:492-523) -----------------------------------------------------------------
    @staticmethod
    def load(model, resume_epoch=None):
        model_path = model.opt.model_path
        if model_path is None:
            name = 'model_latest.pt' if resume_epoch is None else None
            if name is None:
                cands = [f for f in os.listdir(model.save_dir) if f.startswith('model_%03d_' % resume_epoch)]
                name = cands[0]
            model_path = os.path.join(model.save_dir, name)
        state_dict = torch.load(model_path, map_location='cpu', weights_only=False)
        model.epoch = state_dict['epoch']
        model.iterations = state_dict['iterations']
        model.netG.load_state_dict(state_dict['netG'])
        if model.isTrain and 'opt_g' in state_dict:
            model.optimizer_G.load_state_dict(state_dict['opt_g'])
        model._frames_seen = int(state_dict.get('frames_seen', 0))
        print('Resume from epoch %d, iteration %d' % (model.epoch, model.iterations))
        return state_dict

    def state_dict(self):
        return {'netG': {k: v.detach().cpu().clone() for k, v in self.netG.state_dict().items()},
                'opt_g': self.optimizer_G.state_dict(), 'epoch': self.epoch, 'iterations': self.iterations,
                'frames_seen': self._frames_seen}


def eld_model():
    """models/__init__.py:3-4"""
    return ELDModel()
