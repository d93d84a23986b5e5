"""GPU parity of the raw->sRGB kernel (csrc/isp.cu through eld_isp_process) against the oracle and the reference golden."""
import os

import numpy as np
import pytest

from tests.conftest import REPO

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.skip('no GPU')
    return t


def _steps(a, b):
    return np.rint(np.abs(a - b) * 255.0)


def test_isp_matches_reference_golden(torch):
    from eld_b200 import process
    k = np.load(os.path.join(REPO, 'tests', 'golden', 'isp_kat.npz'))
    y = process.process(torch.from_numpy(k['x']).cuda(), k['wb'], k['ccm'], gamma=2.2).cpu().numpy()
    s = _steps(y, k['y'])
    # 8-bit outputs: bit-exact except where powf's last-ulp rounding flips the truncation (tolerance: one level, <= 0.2 %)
    assert s.max() <= 1 and (s > 0).mean() <= 2e-3, (s.max(), (s > 0).mean())


@pytest.mark.parametrize('shape', [(3, 4, 64, 64), (1, 4, 5, 7), (50, 4, 8, 8)])
def test_isp_matches_oracle(torch, shape):
    """vectorised and scalar paths, more frames than one launch holds, values outside [0,1]."""
    from eld_b200 import process
    from oracle import isp_ref
    rs = np.random.RandomState(3)
    n = shape[0]
    x = (rs.rand(*shape) * 1.4 - 0.2).astype(np.float32)
    wb = (1.0 + rs.rand(n, 4)).astype(np.float32)
    ccm = (np.eye(3)[None] * 1.5 + rs.randn(n, 3, 3) * 0.2).astype(np.float32)
    y = process.process(torch.from_numpy(x).cuda(), wb, ccm, gamma=2.2).cpu().numpy()
    ref = isp_ref.process(x, wb, ccm, gamma=2.2)
    s = _steps(y, ref)
    assert s.max() <= 1 and (s > 0).mean() <= 2e-3
    assert y.min() >= 0.0 and y.max() <= 1.0


def test_isp_crf_branch_matches_oracle(torch):
    from eld_b200 import process
    from oracle import isp_ref
    rs = np.random.RandomState(4)
    x = rs.rand(2, 4, 32, 32).astype(np.float32)
    wb = np.array([[2.0, 1.0, 1.5, 1.0]] * 2, np.float32)
    ccm = np.tile(np.eye(3, dtype=np.float32)[None], (2, 1, 1))
    E = np.linspace(0.0, 1.0, 1024, dtype=np.float32)
    fs = np.stack([E ** 0.4, E ** 0.45, E ** 0.5]).astype(np.float32)
    y = process.process(torch.from_numpy(x).cuda(), wb, ccm, CRF=(np.tile(E, (3, 1)), fs)).cpu().numpy()
    ref = isp_ref.process(x, wb, ccm, CRF=(E, fs))
    s = _steps(y, ref)
    assert s.max() <= 1 and (s > 0).mean() <= 2e-3


def test_isp_dataset_item_and_numpy_seam(torch):
    """ISPDataset.__getitem__ (sid_dataset.py:309-312) = clip, raw2rgb_v2, clip; raw2rgb_v2 keeps numpy in / numpy out."""
    from eld_b200 import process
    from oracle import isp_ref
    rs = np.random.RandomState(5)
    x = (rs.rand(4, 16, 16) * 1.2 - 0.1).astype(np.float32)
    wb = np.array([1.9, 1.0, 1.7, 1.0], np.float32)
    ccm = np.array([[1.6, -0.4, -0.2], [-0.3, 1.5, -0.2], [0.0, -0.5, 1.5]], np.float32)
    a = process.raw2rgb_v2(np.clip(x, 0, 1), wb, ccm)
    b = process.isp_dataset_item(torch.from_numpy(x[None]).cuda(), wb[None], ccm[None])[0].cpu().numpy()
    ref = isp_ref.process(np.clip(x, 0, 1)[None], wb[None], ccm[None])[0]
    assert isinstance(a, np.ndarray) and a.shape == (3, 16, 16)
    assert _steps(a, ref).max() <= 1 and _steps(b, ref).max() <= 1


def test_isp_crf_branch_matches_reference_golden(torch):
    """The CRF branch of the kernel against the golden the UNMODIFIED reference produced on its own EMoR curves
    (torchinterp1d -> scipy.interpolate.interp1d, the reference's own yardstick; see tests/test_isp_cpu.py)."""
    from eld_b200 import process
    k = np.load(os.path.join(REPO, 'tests', 'golden', 'isp_crf_kat.npz'))
    y = process.process(torch.from_numpy(k['x']).cuda(), k['wb'], k['ccm'], CRF=(k['E'], k['fs'])).cpu().numpy()
    s = _steps(y, k['y'])
    unsat = k['y'] < 1.0
    assert s[unsat].max() <= 1 and (s[unsat] > 0).mean() <= 5e-3, (s[unsat].max(), (s[unsat] > 0).mean())
    assert s[~unsat].max() <= 1
