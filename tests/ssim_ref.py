"""CPU ORACLE for SSIM (test infrastructure, NOT product code) - the SSIM half of quality_assess.  Only tests/ import it.

    ssim       <- /root/reference/util/index.py:76-81 quality_assess -> skimage.metrics.structural_similarity(
                  Y, X, data_range=255, multichannel=True) with its defaults: win_size 7, gaussian_weights False,
                  use_sample_covariance True, K1 0.01, K2 0.03
                  (third-party scikit-image, not installed: restated from its published algorithm, float64,
                  scipy.ndimage.uniform_filter, crop by (win_size - 1) // 2, mean over the channels)
    ssim_fp32  <- not a reference function: the arithmetic of csrc/eval.cu's eval_ssim_tile_kernel in numpy float32
                  (values less 127.5, direct 7-tap row sums, then direct 7-tap column sums, fp32 formula), to show what
                  fp32 window sums cost

Parity is unpinned by a reference-run golden (skimage cannot be installed); tests/test_ssim_cpu.py pins `ssim` by a
brute-force window loop and closed forms.
"""
import numpy as np
from scipy.ndimage import uniform_filter

WIN = 7


def _check(X, Y):
    X, Y = np.asarray(X), np.asarray(Y)
    if X.shape != Y.shape or X.ndim != 3:
        raise ValueError('ssim: X and Y must be HWC arrays of one shape, got %s and %s' % (X.shape, Y.shape))
    if X.shape[0] < WIN or X.shape[1] < WIN:
        raise ValueError('win_size exceeds image extent: H and W must be >= 7, got %s' % (X.shape[:2],))
    return X, Y


def ssim(X, Y, data_range=255):
    """skimage structural_similarity(X, Y, data_range, multichannel=True) with the defaults, on HWC arrays."""
    X, Y = _check(X, Y)
    pad = (WIN - 1) // 2
    cov_norm = WIN * WIN / (WIN * WIN - 1.0)
    C1, C2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    vals = []
    for ch in range(X.shape[2]):
        x, y = X[..., ch].astype(np.float64), Y[..., ch].astype(np.float64)
        ux, uy = uniform_filter(x, size=WIN), uniform_filter(y, size=WIN)
        uxx, uyy, uxy = uniform_filter(x * x, size=WIN), uniform_filter(y * y, size=WIN), uniform_filter(x * y, size=WIN)
        vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
        S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
        vals.append(S[pad:-pad, pad:-pad].mean())
    return float(np.mean(vals))


def _win_sums_fp32(a, axis):
    n = a.shape[axis] - WIN + 1
    take = (lambda k: a[k:k + n]) if axis == 0 else (lambda k: a[:, k:k + n])
    s = take(0).copy()
    for k in range(1, WIN):
        s += take(k)
    return s


def ssim_fp32(X, Y):
    """the kernel's arithmetic (data_range 255): values shifted by -127.5 (moments about mid-range), fp32 window sums
    in tap order, fp32 formula, double mean"""
    X, Y = _check(X, Y)
    f = np.float32
    inv, cov, k = f(1) / f(49), f(49) / f(48), f(127.5)
    C1, C2 = f(0.01 * 255) * f(0.01 * 255), f(0.03 * 255) * f(0.03 * 255)
    vals = []
    for ch in range(X.shape[2]):
        x, y = X[..., ch].astype(f) - k, Y[..., ch].astype(f) - k
        mx, my, mxx, myy, mxy = [_win_sums_fp32(_win_sums_fp32(q, 1), 0) * inv for q in (x, y, x * x, y * y, x * y)]
        vx, vy, vxy = cov * (mxx - mx * mx), cov * (myy - my * my), cov * (mxy - mx * my)
        ux, uy = mx + k, my + k
        S = ((f(2) * ux * uy + C1) * (f(2) * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))
        vals.append(S.astype(np.float64).mean())
    return float(np.mean(vals))
