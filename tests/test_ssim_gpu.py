"""GPU tests of the device SSIM (csrc/eval.cu eld_eval_ssim, ELDModel.eval_ssim / eval, Engine.eval) against the float64
oracle tests/ssim_ref.py (skimage's structural_similarity restated)."""
import ctypes

import numpy as np
import pytest

from tests import ssim_ref

pytestmark = pytest.mark.gpu

TOL = 2e-6


@pytest.fixture(scope='module')
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no GPU')
    return torch


@pytest.fixture(scope='module')
def model(torch, tmp_path_factory):
    from eld_b200 import models
    m = models.eld_model()
    m.initialize(models.default_opt(name='ssim', checkpoints_dir=str(tmp_path_factory.mktemp('ck'))))
    return m


def _im(x):
    """tensor2im of every frame: [n] HWC float32 arrays, clip(255 v, 0, 255), no rounding"""
    from oracle import eval_ref
    x = x.detach().cpu().numpy()
    return [eval_ref.tensor2im(x[i:i + 1]) for i in range(x.shape[0])]


def _oracle(pred, target):
    return np.array([ssim_ref.ssim(a, b) for a, b in zip(_im(pred), _im(target))])


def _frames(torch, shape, seed):
    """target in [-0.1, 1.1] (the clip at 0 and 255 is exercised) and a noisy prediction of it"""
    g = torch.Generator().manual_seed(seed)
    t = torch.rand(*shape, generator=g) * 1.2 - 0.1
    p = t + 0.1 * torch.randn(*shape, generator=g)
    return p.cuda(), t.cuda()


@pytest.mark.parametrize('shape', [(1, 4, 7, 7), (2, 4, 13, 29), (3, 3, 512, 512), (1, 4, 1424, 2128)])
def test_kernel_matches_the_oracle(torch, model, shape):
    p, t = _frames(torch, shape, sum(shape))
    assert (p < 0).any() and (p > 1).any()
    got = model.eval_ssim(p, t).cpu().numpy()
    want = _oracle(p, t)
    d = np.abs(got - want).max()
    print('max |dSSIM| %s: %.3e' % (shape, d))
    assert d <= TOL, (shape, got, want)
    same = model.eval_ssim(t, t).cpu().numpy()
    assert np.abs(same - 1.0).max() <= 1e-6, same


def test_unaligned_planes(torch, model):
    """w % 4 == 0 but the planes start 4 bytes into their storage: the float4 staging must not be used"""
    p, t = _frames(torch, (1, 4, 40, 272), 9)

    def shifted(a):
        v = torch.empty(a.numel() + 1, device='cuda')[1:].view_as(a)
        v.copy_(a)
        return v
    pv, tv = shifted(p), shifted(t)
    assert pv.data_ptr() % 16 != 0 and tv.data_ptr() % 16 != 0
    got = model.eval_ssim(pv, tv).cpu().numpy()
    assert np.abs(got - _oracle(p, t)).max() <= TOL


def test_batch_frames_are_independent(torch, model):
    p, t = _frames(torch, (3, 4, 64, 96), 5)
    batch = model.eval_ssim(p, t)
    single = torch.cat([model.eval_ssim(p[i:i + 1], t[i:i + 1]) for i in range(3)])
    # the per-plane tile sums are added atomically in double: their order cannot change the f32 result in practice
    assert torch.equal(batch, single), (batch, single)


def test_one_frame_target_is_broadcast(torch, model):
    p, t = _frames(torch, (3, 4, 32, 48), 6)
    got = model.eval_ssim(p, t[:1])
    want = model.eval_ssim(p, t[:1].expand_as(p).contiguous())
    assert torch.equal(got, want)
    assert np.abs(got.cpu().numpy() - _oracle(p, t[:1].expand_as(p))).max() <= TOL


def _eval_case(torch, model, h, w, crop):
    from oracle import eval_ref
    g = torch.Generator().manual_seed(h + w)
    t = torch.rand(1, 4, h, w, generator=g)
    t[0, 0, 100:108, 100:108] = 1.0
    d = {'input': (t * 0.5 + 0.02 * torch.randn(1, 4, h, w, generator=g)).clamp(0, 1), 'target': t, 'fn': ['x']}
    r = model.eval(d, correct=True, crop=crop)
    out = model.output
    xc, tc = d['input'], t
    if crop:
        xc, tc = eval_ref.crop_center(xc, 512, 512), eval_ref.crop_center(tc, 512, 512)
    want = ssim_ref.ssim(_im(out)[0], _im(tc)[0])
    want_in = ssim_ref.ssim(_im(xc)[0], _im(tc)[0])
    print('eval %dx%d crop=%s: |dSSIM| %.3e, |dSSIM_input| %.3e' % (h, w, crop, abs(r['SSIM'] - want), abs(r['SSIM_input'] - want_in)))
    assert abs(r['SSIM'] - want) <= TOL and abs(r['SSIM_input'] - want_in) <= TOL, (r, want, want_in)
    # PSNR keys are those of eval_metrics on the same tensors
    _, psnr, _ = model.eval_metrics(out, tc.cuda())
    _, psnr_in, _ = model.eval_metrics(xc.contiguous().cuda(), tc.cuda())
    assert abs(r['PSNR'] - psnr[0].item()) <= 1e-4 and abs(r['PSNR_input'] - psnr_in[0].item()) <= 1e-4
    want_psnr_in = eval_ref.psnr(_im(xc)[0], _im(tc)[0])
    assert abs(r['PSNR_input'] - want_psnr_in) < 1e-3
    assert np.isfinite(r['SSIM']) and -1.0 <= r['SSIM'] <= 1.0 and 0.0 < r['SSIM_input'] <= 1.0
    return r


def test_eval_reports_ssim_cropped(torch, model):
    r = _eval_case(torch, model, 544, 576, crop=True)
    assert set(r) == {'PSNR', 'PSNR_input', 'SSIM', 'SSIM_input'}


def test_eval_reports_ssim_full_frame(torch, model):
    _eval_case(torch, model, 1424, 2128, crop=False)


def test_engine_eval_averages_ssim(torch, tmp_path):
    """the reference's test loop: res = engine.eval(loader, dataset_name=..., correct=True, crop=False); res['SSIM']"""
    from eld_b200 import models
    from eld_b200.engine import Engine
    eng = Engine(models.default_opt(name='ssim_eng', checkpoints_dir=str(tmp_path), isTrain=False))
    g = torch.Generator().manual_seed(12)
    loader = []
    for i in range(3):
        t = torch.rand(1, 4, 96, 160, generator=g)
        loader.append({'input': (t * 0.3 + 0.01 * torch.randn(1, 4, 96, 160, generator=g)).clamp(0, 1), 'target': t,
                       'fn': ['f%d' % i]})
    res = eng.eval(loader, dataset_name='eld_eval_x', correct=True, crop=False)
    per = [eng.model.eval(d, correct=True, crop=False) for d in loader]
    for k in ('PSNR', 'SSIM', 'SSIM_input'):
        assert abs(res[k] - sum(p[k] for p in per) / 3) <= 1e-6, k
    assert np.isfinite(res['PSNR']) and np.isfinite(res['SSIM']) and 0.0 < res['SSIM_input'] <= 1.0


def test_abi_rejects_bad_shapes_without_launching(torch, model):
    from eld_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(2 * 4 * 8 * 8, device='cuda')
    s = torch.zeros(8, dtype=torch.float64, device='cuda')
    o = torch.zeros(2, device='cuda')
    ctx = _lib.ctx(0)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    before = _lib.launch_count(0)
    cases = [(x.data_ptr(), x.data_ptr(), 2, 4, 6, 8, s.data_ptr(), o.data_ptr()),
             (x.data_ptr(), x.data_ptr(), 2, 4, 8, 6, s.data_ptr(), o.data_ptr()),
             (x.data_ptr(), x.data_ptr(), 2, 0, 8, 8, s.data_ptr(), o.data_ptr()),
             (x.data_ptr(), x.data_ptr(), 0, 4, 8, 8, s.data_ptr(), o.data_ptr()),
             (None, x.data_ptr(), 2, 4, 8, 8, s.data_ptr(), o.data_ptr()),
             (x.data_ptr(), None, 2, 4, 8, 8, s.data_ptr(), o.data_ptr()),
             (x.data_ptr(), x.data_ptr(), 2, 4, 8, 8, None, o.data_ptr()),
             (x.data_ptr(), x.data_ptr(), 2, 4, 8, 8, s.data_ptr(), None)]
    for a in cases:
        assert lib.eld_eval_ssim(ctx, *a, st) == -1, a
    assert lib.eld_eval_ssim(ctx, *cases[0], st) == -1 and b'7 x 7' in lib.eld_last_error()
    assert _lib.launch_count(0) == before
    assert lib.eld_eval_ssim(ctx, x.data_ptr(), x.data_ptr(), 2, 4, 8, 8, s.data_ptr(), o.data_ptr(), st) == 0
    assert _lib.launch_count(0) == before + 2
    assert (o - 1).abs().max().item() <= 1e-6
