"""Bit-exactness of the two cell-level rewrites of the tiled row forward (csrc/probit_rows.cu):

* probit_math.cuh::erf_dual, the erf of the faithful forward's probit_E on the device, must return libdevice erff's bits
  for every one of the 2^32 fp32 inputs;
* common.cuh::warp_sum_transposed, which reduces the forward's per-(sample pair, chunk) sums several at a time, must give
  each total the plain warp_sum butterfly's bits, NaN, +-Inf and +-0 included.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _stream():
    return C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)


def test_erf_bits_every_fp32():
    from mpvae_b200 import _lib
    chunk = 1 << 28
    out = torch.empty(chunk, dtype=torch.float32, device=DEV)
    ref = torch.empty_like(out)
    bad = 0
    for start in range(0, 1 << 32, chunk):
        bits = torch.arange(start - (1 << 31), start - (1 << 31) + chunk, dtype=torch.int64, device=DEV).to(torch.int32)
        x = bits.view(torch.float32)
        _lib.check(_lib.lib().mpvae_test_erf(C.c_void_p(x.data_ptr()), C.c_void_p(out.data_ptr()), C.c_void_p(ref.data_ptr()),
                                             chunk, _stream()), "mpvae_test_erf")
        bad += int((out.view(torch.int32) != ref.view(torch.int32)).sum())
        del bits, x
    assert bad == 0, f"{bad} inputs where erf_dual differs from erff"


def _specials(dtype):
    return np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -1.0, np.finfo(dtype).max, -np.finfo(dtype).max,
                     np.finfo(dtype).tiny, np.finfo(dtype).smallest_subnormal], dtype=dtype)


@pytest.mark.parametrize("fp64", [False, True])
def test_warp_sum_transposed_bits(fp64):
    from mpvae_b200 import _lib
    dtype, tdtype, n = (np.float64, torch.float64, 4) if fp64 else (np.float32, torch.float32, 8)
    rng = np.random.default_rng(7 + fp64)
    groups = 20000
    # mixed magnitudes, so that the order of the adds shows in the low bits
    x = (rng.standard_normal((groups, 32, n)) * np.exp2(rng.integers(-30, 30, (groups, 32, n)))).astype(dtype)
    # rare specials in most groups (a single NaN / Inf decides the total), and groups of special values only
    sp = _specials(dtype)
    few = rng.random((groups, 32, n)) < 0.002
    x[few] = rng.choice(sp, int(few.sum()))
    x[-500:] = rng.choice(sp, (500, 32, n))
    x[-600:-500] = rng.choice(np.array([0.0, -0.0], dtype=dtype), (100, 32, n))
    inp = torch.from_numpy(x).to(DEV)
    out = torch.full((groups, n), 7.0, dtype=tdtype, device=DEV)
    ref = torch.full_like(out, -7.0)
    _lib.check(_lib.lib().mpvae_test_warp_sum(C.c_void_p(inp.data_ptr()), C.c_void_p(out.data_ptr()), C.c_void_p(ref.data_ptr()),
                                              groups, int(fp64), _stream()), "mpvae_test_warp_sum")
    torch.cuda.synchronize()
    itype = torch.int64 if fp64 else torch.int32
    o, r = out.view(itype), ref.view(itype)
    assert torch.equal(o, r), f"{int((o != r).sum())} of {o.numel()} totals differ"
    assert torch.isnan(ref).any() and torch.isinf(ref).any()   # the specials did reach the totals
