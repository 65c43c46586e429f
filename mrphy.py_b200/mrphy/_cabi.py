"""ctypes binding of libmrphy_b200.so (C ABI declared in include/mrphy_b200.h).

No torch types cross this boundary: tensors are passed as ``data_ptr()`` + element strides, the
stream as ``torch.cuda.current_stream().cuda_stream``.  The library is loaded lazily; if it is
missing the hot path raises -- there is no other implementation to fall back to.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MRPHY_B200_LIB') or os.path.join(os.path.dirname(_HERE), 'libmrphy_b200.so')

MRPHY_F32, MRPHY_F64 = 0, 1
FLAG_TRIG_PRECISE, FLAG_NEED_GMI, FLAG_RF_COIL_DIM, FLAG_NEED_GBEFF, FLAG_TRIG_FAST_BWD = 1, 2, 4, 8, 16
FLAG_SKIP_GRF, FLAG_SKIP_GGR, FLAG_ZERO_GRAD_TAIL = 32, 64, 128
ABI_VERSION = 7

c_i32, c_i64, c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p


class Param(ctypes.Structure):
    _fields_ = [('ptr', c_vp), ('sn', c_i64), ('sm', c_i64), ('f64', c_i32), ('_pad', c_i32)]


class FusedArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('flags', c_i32), ('N', c_i32), ('nM', c_i32), ('nT', c_i32), ('nC', c_i32),
        ('K', c_i32), ('_pad', c_i32),
        ('Mi', c_vp), ('Mi_sn', c_i64), ('Mi_sm', c_i64),
        ('rf', c_vp), ('rf_sn', c_i64), ('rf_sx', c_i64), ('rf_st', c_i64), ('rf_sc', c_i64),
        ('gr', c_vp), ('gr_sn', c_i64), ('gr_sx', c_i64), ('gr_st', c_i64),
        ('loc', c_vp), ('loc_sn', c_i64), ('loc_sm', c_i64),
        ('b1', c_vp), ('b1_sn', c_i64), ('b1_sm', c_i64),
        ('df', Param), ('T1', Param), ('T2', Param), ('gamma', Param), ('dt', Param),
        ('Mo', c_vp), ('ckpt', c_vp), ('wave', c_vp),
        ('gMo', c_vp), ('gMo_sn', c_i64), ('gMo_sm', c_i64),
        ('gMi', c_vp), ('grf', c_vp), ('ggr', c_vp), ('partials', c_vp),
        ('every', c_i32), ('nR', c_i32), ('Mt', c_vp), ('gMt', c_vp),
        ('gloc', c_vp), ('gsz', c_vp), ('gb1', c_vp),
        ('design', c_vp),
    ]


class BeffArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('flags', c_i32), ('N', c_i32), ('nM', c_i32), ('nT', c_i32), ('K', c_i32),
        ('Mi', c_vp), ('Mi_sn', c_i64), ('Mi_sm', c_i64),
        ('Beff', c_vp), ('B_sn', c_i64), ('B_sm', c_i64), ('B_st', c_i64),
        ('T1', Param), ('T2', Param), ('gamma', Param), ('dt', Param),
        ('Mo', c_vp), ('ckpt', c_vp),
        ('gMo', c_vp), ('gMo_sn', c_i64), ('gMo_sm', c_i64),
        ('gMi', c_vp), ('gBeff', c_vp),
    ]


class RfGr2BeffArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('flags', c_i32), ('N', c_i32), ('nM', c_i32), ('nT', c_i32), ('nC', c_i32),
        ('rf', c_vp), ('rf_sn', c_i64), ('rf_sx', c_i64), ('rf_st', c_i64), ('rf_sc', c_i64),
        ('gr', c_vp), ('gr_sn', c_i64), ('gr_sx', c_i64), ('gr_st', c_i64),
        ('loc', c_vp), ('loc_sn', c_i64), ('loc_sm', c_i64),
        ('b1', c_vp), ('b1_sn', c_i64), ('b1_sm', c_i64),
        ('df', Param), ('gamma', Param),
        ('Beff', c_vp), ('gBeff', c_vp), ('grf', c_vp), ('ggr', c_vp), ('partials', c_vp),
        ('gloc', c_vp), ('gsz', c_vp), ('gb1', c_vp),
    ]


class Beff2abArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('flags', c_i32), ('N', c_i32), ('nM', c_i32), ('nT', c_i32), ('K', c_i32),
        ('Beff', c_vp), ('B_sn', c_i64), ('B_sm', c_i64),
        ('E1', Param), ('E2', Param), ('gamma', Param), ('dt', Param),
        ('A', c_vp), ('B', c_vp), ('ckpt', c_vp), ('gA', c_vp), ('gB', c_vp), ('gBeff', c_vp), ('gP', c_vp),
    ]


class Beff2uphiArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('adjoint', c_i32), ('N', c_i32), ('nM', c_i32),
        ('beff', c_vp), ('b_sn', c_i64), ('b_sm', c_i64),
        ('g', Param),
        ('U', c_vp), ('Phi', c_vp), ('gU', c_vp), ('gPhi', c_vp), ('gbeff', c_vp), ('gg', c_vp),
    ]


class FreePrecArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('adjoint', c_i32), ('N', c_i32), ('nM', c_i32),
        ('Mi', c_vp), ('Mi_sn', c_i64), ('Mi_sm', c_i64),
        ('dur', Param), ('T1', Param), ('T2', Param), ('df', Param),
        ('Mo', c_vp),
    ]


class ReparamArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('adjoint', c_i32), ('N', c_i32), ('nT', c_i32), ('nC', c_i32), ('rf_kind', c_i32),
        ('gr_kind', c_i32), ('_pad', c_i32),
        ('rho', c_vp), ('theta', c_vp), ('rfmax', c_vp), ('rfmax_sn', c_i64), ('rfmax_sc', c_i64),
        ('ts', c_vp), ('smax', c_vp), ('smax_sn', c_i64), ('smax_sx', c_i64),
        ('dt', Param),
        ('rf', c_vp), ('gr', c_vp), ('grf', c_vp), ('ggr', c_vp), ('grho', c_vp), ('gtheta', c_vp), ('gts', c_vp),
    ]


class MaskArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('N', c_i32), ('fill_zero', c_i32), ('_pad', c_i32), ('nOut', c_i64), ('nIn', c_i64),
        ('inner', c_i64),
        ('idx', c_vp), ('inp', c_vp), ('out', c_vp),
    ]


class ClampArgs(ctypes.Structure):
    _fields_ = [
        ('dtype', c_i32), ('adjoint', c_i32), ('kind', c_i32), ('N', c_i32), ('nT', c_i32), ('nC', c_i32),
        ('x', c_vp), ('lim', c_vp), ('lim_sn', c_i64), ('lim_sc', c_i64), ('eps', ctypes.c_double),
        ('g', c_vp), ('out', c_vp),
    ]


EXPORTS = {   # name -> (restype, argtypes); tests check every symbol include/mrphy_b200.h declares
    'mrphy_abi_version': (ctypes.c_int, []),
    'mrphy_last_error': (ctypes.c_char_p, []),
    'mrphy_sizeof_args': (ctypes.c_size_t, [ctypes.c_int]),
    'mrphy_last_launch_count': (ctypes.c_int, []),
    'mrphy_device_sm_count': (ctypes.c_int, [ctypes.c_int]),
    'mrphy_kernel_timing': (ctypes.c_int, [ctypes.c_int]),
    'mrphy_last_kernel_ms': (ctypes.c_float, []),
    'mrphy_fused_ckpt_elems': (ctypes.c_size_t, [ctypes.POINTER(FusedArgs)]),
    'mrphy_fused_wave_elems': (ctypes.c_size_t, [ctypes.POINTER(FusedArgs)]),
    'mrphy_fused_partial_elems': (ctypes.c_size_t, [ctypes.POINTER(FusedArgs)]),
    'mrphy_blochsim_fused_fwd': (ctypes.c_int, [ctypes.POINTER(FusedArgs), c_vp]),
    'mrphy_blochsim_fused_bwd': (ctypes.c_int, [ctypes.POINTER(FusedArgs), ctypes.c_int, c_vp]),
    'mrphy_beff_ckpt_elems': (ctypes.c_size_t, [ctypes.POINTER(BeffArgs)]),
    'mrphy_blochsim_beff_fwd': (ctypes.c_int, [ctypes.POINTER(BeffArgs), c_vp]),
    'mrphy_blochsim_beff_bwd': (ctypes.c_int, [ctypes.POINTER(BeffArgs), c_vp]),
    'mrphy_rfgr2beff': (ctypes.c_int, [ctypes.POINTER(RfGr2BeffArgs), c_vp]),
    'mrphy_rfgr2beff_partial_elems': (ctypes.c_size_t, [ctypes.POINTER(RfGr2BeffArgs)]),
    'mrphy_rfgr2beff_bwd': (ctypes.c_int, [ctypes.POINTER(RfGr2BeffArgs), c_vp]),
    'mrphy_rfgr2beff_spin_grads': (ctypes.c_int, [ctypes.POINTER(RfGr2BeffArgs), c_vp]),
    'mrphy_beff2ab_ckpt_elems': (ctypes.c_size_t, [ctypes.POINTER(Beff2abArgs)]),
    'mrphy_beff2ab': (ctypes.c_int, [ctypes.POINTER(Beff2abArgs), c_vp]),
    'mrphy_beff2ab_bwd': (ctypes.c_int, [ctypes.POINTER(Beff2abArgs), c_vp]),
    'mrphy_beff2uphi': (ctypes.c_int, [ctypes.POINTER(Beff2uphiArgs), c_vp]),
    'mrphy_freeprec': (ctypes.c_int, [ctypes.POINTER(FreePrecArgs), c_vp]),
    'mrphy_design_waveform': (ctypes.c_int, [ctypes.POINTER(ReparamArgs), c_vp]),
    'mrphy_mask_copy': (ctypes.c_int, [ctypes.POINTER(MaskArgs), c_vp]),
    'mrphy_clamp_waveform': (ctypes.c_int, [ctypes.POINTER(ClampArgs), c_vp]),
}

_lib = None
_lock = threading.Lock()


def lib():
    """The loaded library; raises RuntimeError (never falls back) when it is not built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH) and 'MRPHY_B200_LIB' not in os.environ:
                    _try_build()
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f'mrphy (B200): {LIB_PATH} is not built. Run `python mrphy.py_b200/build.py` '
                        '(nvcc, sm_100a). There is no CPU or PyTorch fallback for the Bloch-simulation path.')
                L = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in EXPORTS.items():
                    fn = getattr(L, name)
                    fn.restype, fn.argtypes = res, args
                if L.mrphy_abi_version() != ABI_VERSION:
                    raise RuntimeError(f'mrphy (B200): ABI version mismatch: library {L.mrphy_abi_version()} '
                                       f'!= binding {ABI_VERSION}; rebuild with mrphy.py_b200/build.py')
                mirrors = (Param, FusedArgs, BeffArgs, RfGr2BeffArgs, Beff2abArgs, Beff2uphiArgs, FreePrecArgs, ReparamArgs,
                           MaskArgs, ClampArgs)
                for which, cls in enumerate(mirrors):
                    if L.mrphy_sizeof_args(which) != ctypes.sizeof(cls):
                        raise RuntimeError(f'mrphy (B200): layout of {cls.__name__} ({ctypes.sizeof(cls)} B) differs from '
                                           f'the library ({L.mrphy_sizeof_args(which)} B); rebuild with mrphy.py_b200/build.py')
                _lib = L
    return _lib


def _try_build():
    """Compile the library in-tree when it is missing and nvcc is on the box (never a non-CUDA substitute)."""
    import importlib.util
    import shutil
    if not (shutil.which('nvcc') or os.path.exists('/usr/local/cuda/bin/nvcc')):
        return
    try:
        spec = importlib.util.spec_from_file_location('mrphy_build', os.path.join(os.path.dirname(_HERE), 'build.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    except Exception as e:   # surfaced by the RuntimeError below
        import warnings
        warnings.warn(f'mrphy (B200): building {LIB_PATH} failed: {e}')


def check(rc, what):
    if rc != 0:
        msg = lib().mrphy_last_error().decode(errors='replace')
        raise RuntimeError(f'mrphy (B200): {what} failed with status {rc}: {msg}')


# launches issued by this process through the C ABI (bench.py reports it as gpu_launches)
launch_counter = 0


def count_launches():
    global launch_counter
    launch_counter += lib().mrphy_last_launch_count()
