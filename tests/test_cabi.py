"""The C-ABI library loads and exports every symbol include/mrphy_b200.h declares (no compute calls)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, 'include', 'mrphy_b200.h')


@pytest.fixture(scope='module')
def cabi():
    import importlib.util
    import sys
    spec = importlib.util.spec_from_file_location('mrphy_build', os.path.join(ROOT, 'mrphy.py_b200', 'build.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()                      # no-op when the in-tree .so is fresh
    from mrphy import _cabi
    return _cabi


def declared_functions():
    src = re.sub(r'/\*.*?\*/', '', open(HDR).read(), flags=re.S)
    return sorted(set(re.findall(r'\b(mrphy_[a-z0-9_]+)\s*\(', src)))


def test_header_symbols_exported(cabi):
    L = ctypes.CDLL(cabi.LIB_PATH)
    names = declared_functions()
    assert len(names) >= 12
    for n in names:
        assert hasattr(L, n), f'{n} declared in include/mrphy_b200.h but not exported'
    assert set(names) == set(cabi.EXPORTS), 'python binding and header disagree'


def test_abi_version_and_arg_struct_sizes(cabi):
    L = cabi.lib()
    assert L.mrphy_abi_version() == cabi.ABI_VERSION
    # struct sizes must match the C definition (all 8-byte aligned fields)
    assert ctypes.sizeof(cabi.Param) == 32
    assert ctypes.sizeof(cabi.FusedArgs) == 8 * 4 + 8 * 3 + 8 * 5 + 8 * 4 + 8 * 3 + 8 * 3 + 32 * 5 + 8 * 3 + 8 * 3 + 8 * 4 + \
        4 * 2 + 8 * 2 + 8 * 3 + 8                    # options: record, per-spin gradients, design tail
    assert ctypes.sizeof(cabi.BeffArgs) == 6 * 4 + 8 * 3 + 8 * 4 + 32 * 4 + 8 * 2 + 8 * 3 + 8 * 2
    # ... and the C side agrees with every ctypes mirror (the loader checks the same and refuses a mismatch)
    for which, cls in enumerate((cabi.Param, cabi.FusedArgs, cabi.BeffArgs, cabi.RfGr2BeffArgs, cabi.Beff2abArgs,
                                 cabi.Beff2uphiArgs, cabi.FreePrecArgs, cabi.ReparamArgs, cabi.MaskArgs, cabi.ClampArgs)):
        assert L.mrphy_sizeof_args(which) == ctypes.sizeof(cls), cls.__name__
    assert L.mrphy_sizeof_args(99) == 0


def test_sizing_entry_points(cabi):
    L = cabi.lib()
    a = cabi.FusedArgs()
    a.dtype, a.N, a.nM, a.nT, a.nC, a.K = cabi.MRPHY_F32, 2, 1000, 1000, 1, 64
    a.b1 = 1  # non-null: per-coil path
    assert L.mrphy_fused_ckpt_elems(a) == 2 * 15 * 3 * 1000          # ceil(1000/64)-1 = 15 checkpoints
    assert L.mrphy_fused_wave_elems(a) == 2 * 16 * 5 * 64
    # ceil(1000/128) = 8 CTAs per batch entry, plus the backward's scheduling ints (264 + 8) and the epilogue's finished-CTA
    # counters (one per batch entry) behind the partial sums
    assert L.mrphy_fused_partial_elems(a) == 2 * 8 * 5 * 1000 + 264 + 8 + 2
    a.K = 0
    assert L.mrphy_fused_ckpt_elems(a) == 0 and b'K must be' in L.mrphy_last_error()


@pytest.mark.parametrize('nC,K,nT', [(1, 64, 1000), (2, 16, 50), (3, 7, 33), (8, 64, 64), (16, 48, 100),
                                      (8, 32, 100), (4, 16, 50), (16, 24, 70), (5, 1, 9)])   # K <= 32, >= 3 coils: tensor-core operand tiles
def test_fused_fwd_fake_matches_sizing_calls(cabi, nC, K, nT):
    """The torch.library fake (shape-only) implementation must allocate what the C sizing entry points ask for."""
    import torch
    from mrphy import _ops
    N, nM = 2, 300
    a = cabi.FusedArgs()
    a.dtype, a.N, a.nM, a.nT, a.nC, a.K = cabi.MRPHY_F32, N, nM, nT, nC, K
    a.b1 = 1
    L = cabi.lib()
    m = dict(device='meta')
    rf = torch.empty(N, 2, nT, nC, **m) if nC > 1 else torch.empty(N, 2, nT, **m)
    b1 = torch.empty(N, nM, 2, nC, **m)
    Mo, _, ckpt, wave = _ops._fake_blochsim_fused_fwd(torch.empty(N, nM, 3, **m), rf, torch.empty(N, 3, nT, **m),
                                                      torch.empty(N, nM, 3, **m), None, b1, None, None, None, None, K, 0, 0)
    assert tuple(Mo.shape) == (N, nM, 3)
    assert ckpt.numel() == max(L.mrphy_fused_ckpt_elems(a), 1)
    assert wave.numel() == L.mrphy_fused_wave_elems(a)


def test_fails_loudly_without_gpu_or_on_cpu_tensors(cabi):
    import torch
    import mrphy
    from mrphy import sims, mobjs
    M = torch.zeros(1, 4, 3)
    B = torch.zeros(1, 4, 8, 3)
    with pytest.raises(RuntimeError, match='CUDA-only'):
        sims.blochsim(M, B)
    cube, pulse = mobjs.Examples.spincube(), mobjs.Examples.pulse()
    with pytest.raises(RuntimeError, match='CUDA-only'):
        cube.applypulse(pulse)
    if not torch.cuda.is_available():
        a = cabi.FusedArgs()
        a.dtype, a.N, a.nM, a.nT, a.nC, a.K = 0, 1, 4, 8, 1, 8
        for f in ('Mi', 'rf', 'gr', 'loc', 'Mo', 'ckpt', 'wave'):
            setattr(a, f, 256)
        a.gamma.ptr, a.dt.ptr = 256, 256
        rc = cabi.lib().mrphy_blochsim_fused_fwd(a, None)
        assert rc == -2 and cabi.lib().mrphy_last_error() != b''     # MRPHY_ERR_CUDA, never a silent fallback
