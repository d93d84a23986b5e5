"""ctypes binding of libeld_b200.so (the C ABI in include/eld_b200.h).

The library is the product; there is NO CPU fallback: if the shared object is missing or the
machine has no CUDA device, every compute call raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libeld_b200.so')

MODEL_BITS = {'P': 0x01, 'p': 0x02, 'g': 0x04, 'G': 0x08, 'B': 0x10, 'R': 0x20, 'U': 0x40}
DT_U16, DT_F32, DT_BF16 = 0, 1, 2


class EldError(RuntimeError):
    pass


class NoiseParams(ctypes.Structure):
    """eld_noise_params (48 bytes)."""
    _fields_ = [('K', ctypes.c_float), ('g_scale', ctypes.c_float), ('G_scale', ctypes.c_float),
                ('G_lambda', ctypes.c_float), ('R_scale', ctypes.c_float), ('q_step', ctypes.c_float),
                ('saturation', ctypes.c_float), ('ratio', ctypes.c_float), ('color_bias', ctypes.c_float * 4)]


_lib = None


def _declare(lib):
    c = ctypes
    vp, i32, u32, u64, f32 = c.c_void_p, c.c_int, c.c_uint32, c.c_uint64, c.c_float
    lib.eld_abi_version.restype = i32
    lib.eld_last_error.restype = c.c_char_p
    lib.eld_ctx_create.argtypes = [i32, c.POINTER(vp)]
    lib.eld_ctx_destroy.argtypes = [vp]
    lib.eld_ctx_destroy.restype = None
    lib.eld_launch_count.argtypes = [vp]
    lib.eld_launch_count.restype = c.c_int64
    lib.eld_noise_packed.argtypes = [vp, vp, vp, i32, i32, i32, c.POINTER(NoiseParams), u32, u64, u64, i32, vp]
    lib.eld_noise_mosaic.argtypes = [vp, vp, i32, f32, f32, vp, vp, i32, i32, i32, c.POINTER(NoiseParams),
                                     u32, u64, u64, i32, vp]
    lib.eld_noise_packed_u16.argtypes = [vp, vp, f32, vp, vp, i32, i32, i32, c.POINTER(NoiseParams), u32, u64, u64, i32, vp]
    lib.eld_isp_process.argtypes = [vp, vp, vp, i32, i32, i32, c.POINTER(c.c_float), c.POINTER(c.c_float), f32, vp, vp, i32, vp]
    lib.eld_noise_packed_aug.argtypes = [vp, vp, vp, vp, i32, i32, i32, c.POINTER(NoiseParams), u32, u64, u64, i32,
                                         c.POINTER(c.c_uint8), vp]
    lib.eld_eval_correct_psnr.argtypes = [vp, vp, vp, vp, i32, c.c_size_t, i32, vp, vp, vp, vp]
    lib.eld_eval_ssim.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp]
    from . import _unet_abi
    _unet_abi.declare(lib)


def load():
    """Load libeld_b200.so (once).  Raises EldError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EldError('%s not found - run `python -m eld_b200.build` (or __graft_entry__.build()); '
                           'there is no CPU fallback' % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        _declare(lib)
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        raise EldError('%s failed (%d): %s' % (what, rc, load().eld_last_error().decode('utf-8', 'replace')))


_ctxs = {}


def ctx(device=0):
    """One eld_ctx per device, created lazily."""
    if device not in _ctxs:
        lib = load()
        h = ctypes.c_void_p()
        check(lib.eld_ctx_create(int(device), ctypes.byref(h)), 'eld_ctx_create')
        _ctxs[device] = h
    return _ctxs[device]


def launch_count(device=0):
    return int(load().eld_launch_count(ctx(device)))


def model_mask(model):
    """Reference semantics (noise.py:158-166): substring tests for 'P', 'p', 'g' on the model string; 'P' wins over
    'p'; every other character is ignored (so the README's names 'G+P', 'G+P*' mean what they mean in the reference).
    The paper-restated terms - G (Tukey-lambda), B (colour bias), R (row), U (quantisation), NOT in the reference -
    are an explicit opt-in: the string must start with 'ELD:' (e.g. 'ELD:P+G+B+R+U')."""
    full = is_full_model(model)
    body = model[4:] if full else model
    m = 0
    if 'P' in body:
        m |= MODEL_BITS['P']
    elif 'p' in body:
        m |= MODEL_BITS['p']
    for ch in ('gGBRU' if full else 'g'):
        if ch in body:
            m |= MODEL_BITS[ch]
    return m


def is_full_model(model):
    return model.startswith('ELD:')
