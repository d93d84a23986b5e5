"""The SSIM oracle (tests/ssim_ref.py, skimage's structural_similarity restated) against a brute-force window loop and
closed forms, and the fp32 arithmetic of csrc/eval.cu's SSIM kernel against the float64 oracle - no GPU."""
import numpy as np
import pytest

from tests import ssim_ref

C1, C2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2


def _brute(X, Y):
    """every interior 7x7 window, float64, sample covariance: the definition written out"""
    H, W, C = X.shape
    vals = []
    for c in range(C):
        s = []
        for i in range(H - 6):
            for j in range(W - 6):
                a = X[i:i + 7, j:j + 7, c].astype(np.float64).ravel()
                b = Y[i:i + 7, j:j + 7, c].astype(np.float64).ravel()
                ux, uy = a.mean(), b.mean()
                vx, vy = np.var(a, ddof=1), np.var(b, ddof=1)
                vxy = np.sum((a - ux) * (b - uy)) / 48.0
                s.append((2 * ux * uy + C1) * (2 * vxy + C2) / ((ux * ux + uy * uy + C1) * (vx + vy + C2)))
        vals.append(np.mean(s))
    return float(np.mean(vals))


def _pair(rng, shape, noise=0.1):
    X = np.clip(rng.rand(*shape) * 255.0, 0, 255).astype(np.float32)
    Y = np.clip(X + noise * 255.0 * rng.randn(*shape), 0, 255).astype(np.float32)
    return X, Y


@pytest.mark.parametrize('shape', [(13, 17, 2), (9, 30, 3)])
def test_oracle_equals_brute_force_windows(shape):
    X, Y = _pair(np.random.RandomState(1), shape)
    assert abs(ssim_ref.ssim(X, Y) - _brute(X, Y)) <= 1e-12


def test_closed_forms():
    rng = np.random.RandomState(2)
    X, Y = _pair(rng, (20, 23, 4))
    assert abs(ssim_ref.ssim(X, X) - 1.0) <= 1e-12
    assert ssim_ref.ssim(X, Y) == ssim_ref.ssim(Y, X)
    for a, b in ((10.0, 200.0), (0.0, 255.0), (37.5, 37.5), (128.0, 3.0)):
        A, B = np.full((11, 9, 3), a, np.float32), np.full((11, 9, 3), b, np.float32)
        # constant planes: every variance is 0, so the contrast-structure factor is C2 / C2
        assert abs(ssim_ref.ssim(A, B) - (2 * a * b + C1) / (a * a + b * b + C1)) <= 1e-12


def test_fp32_window_sums_are_accurate_on_a_full_eld_frame():
    """the kernel sums its 7x7 windows in fp32 about mid-range (uxx - ux^2 cancels): on a full packed ELD frame
    (1424 x 2128 x 4) the frame's SSIM stays within 1e-6 of the float64 oracle, bright and dark, clean and noisy"""
    rng = np.random.RandomState(3)
    yy, xx = np.mgrid[0:1424, 0:2128].astype(np.float32)
    base = 0.5 + 0.4 * np.sin(xx / 37.0)[..., None] * np.cos(yy / 23.0)[..., None] * np.ones(4, np.float32)
    for level, noise in ((1.0, 0.02), (1.0, 0.002), (0.05, 0.002), (1.0, 0.2)):
        clean = np.clip(base * level, 0, 1)
        noisy = clean + noise * rng.randn(*clean.shape).astype(np.float32)
        X, Y = np.clip(noisy * 255.0, 0, 255).astype(np.float32), np.clip(clean * 255.0, 0, 255).astype(np.float32)
        want, got = ssim_ref.ssim(X, Y), ssim_ref.ssim_fp32(X, Y)
        assert abs(got - want) <= 1e-6, (level, noise, got, want)


@pytest.mark.parametrize('shape', [(6, 20, 4), (20, 6, 4), (6, 6, 1)])
def test_rejects_planes_smaller_than_the_window(shape):
    X = np.zeros(shape, np.float32)
    with pytest.raises(ValueError):
        ssim_ref.ssim(X, X)
