"""CPU: the power-of-two operand scales of the tcgen05 split-precision contraction (csrc/common.cuh, __host__ __device__)
compiled for the host and swept over every fp32 exponent.

An fp32 operand is split into two fp16 pieces of x * s with s = 2^k chosen from the tensor's max |x|; the GEMM epilogue
multiplies the accumulated products by 2^-(ka + kb), as two powers of two.  What must hold:
  * every maximum from 2^-112 up to the largest finite fp32 is scaled into [2^14, 2^15), one binade under the fp16 maximum;
  * 0, Inf and NaN give s = 1 (the pieces are the values themselves);
  * descaling is exact whenever the true descaled value is an fp32 normal, for every pair of exponents, and where the
    whole factor 2^-(ka + kb) is an fp32 normal it is the single product acc * 2^-(ka + kb) the epilogue always formed.
No GPU: g++ and the CUDA headers (common.cuh includes cuda_runtime.h)."""
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host", "contract_scale_host.cpp")
CUDA_INC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


@pytest.fixture(scope="module")
def scale_binary(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("CUDA headers not available")
    out = str(tmp_path_factory.mktemp("scale") / "contract_scale_host")
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-ffp-contract=off", "-I", CUDA_INC, "-o", out, SRC])
    return out


def run(binary, a_bits, b_bits, acc_bits):
    recs = np.stack([a_bits, b_bits, acc_bits], axis=1).astype(np.uint64)
    text = f"{len(recs)}\n" + "\n".join(f"{a} {b} {c}" for a, b, c in recs) + "\n"
    res = subprocess.run([binary], input=text, capture_output=True, text=True, check=True)
    out = np.array([ln.split() for ln in res.stdout.strip().splitlines()], dtype=np.int64)
    f = lambda col: out[:, col].astype(np.uint32).view(np.float32)
    return {"ka": out[:, 0], "kb": out[:, 1], "sa": f(2), "sb": f(3), "main": f(4), "extra": f(5), "out": f(6)}


def bits(x):
    return np.asarray(x, dtype=np.float32).view(np.uint32)


def test_every_finite_maximum_scales_into_one_binade_under_the_fp16_maximum(scale_binary):
    # every exponent field of a finite fp32, with the smallest and the largest mantissa
    fields = np.arange(0, 255, dtype=np.uint32)
    maxima = np.concatenate([(fields << 23) | 1, (fields << 23) | 0x7FFFFF]).astype(np.uint32)
    r = run(scale_binary, maxima, maxima, np.zeros_like(maxima))
    m = maxima.view(np.float32).astype(np.float64)
    assert np.array_equal(r["sa"].astype(np.float64), np.ldexp(1.0, r["ka"])), "the scale is 2^k"
    scaled = m * np.ldexp(1.0, r["ka"])                                   # exact in fp64
    supported = m >= 2.0 ** -112
    assert supported.sum() == 2 * (255 - 15)
    assert np.all((scaled[supported] >= 2.0 ** 14) & (scaled[supported] < 2.0 ** 15)), m[supported][
        (scaled[supported] < 2.0 ** 14) | (scaled[supported] >= 2.0 ** 15)]
    # below 2^-112 the scale stops growing (s = 2^126, so that 1 / s is still an fp32 normal): the maximum is scaled to
    # less, never to more
    assert np.all(r["ka"][~supported] == 126) and np.all(scaled[~supported] < 2.0 ** 14)
    # s and 1 / s are fp32 normals for every input
    assert r["ka"].min() >= -126 and r["ka"].max() <= 126
    # the fp16 hi piece of the maximum is finite: the largest fp16 is 65504
    assert np.all(scaled.astype(np.float32).astype(np.float16) <= 65504.0)


def test_zero_inf_and_nan_fall_back_to_scale_one(scale_binary):
    specials = bits([0.0, -0.0, np.inf, -np.inf, np.nan]).copy()
    specials = np.concatenate([specials, np.array([0x7FC00001, 0xFFFFFFFF, 0x7F800001], dtype=np.uint32)])
    r = run(scale_binary, specials, specials, bits(np.full(len(specials), 3.0)))
    assert np.all(r["ka"] == 0) and np.all(r["sa"] == 1.0)
    assert np.all(r["main"] == 1.0) and np.all(r["extra"] == 1.0) and np.all(r["out"] == 3.0)


def test_descaling_is_exact_for_every_pair_of_exponents(scale_binary):
    """All 256 x 256 exponent fields of the two maxima (denormals, Inf / NaN included), against accumulated values from
    tiny to the largest a K = 2^20 product of scaled pieces can reach."""
    fields = np.arange(256, dtype=np.uint32)
    ea, eb = np.meshgrid(fields, fields, indexing="ij")
    a_bits = ((ea.ravel() << 23) | 0x400000).astype(np.uint32)          # 1.5 * 2^e (NaN for the field 255)
    b_bits = ((eb.ravel() << 23) | 0x123457).astype(np.uint32)
    accs = np.array([1.0, -1.5 * 2.0 ** 29, 1.25 * 2.0 ** -20, 3.0 * 2.0 ** 40, -(2.0 ** 50) * 1.75, 2.0 ** -100], dtype=np.float32)
    A = np.repeat(a_bits, len(accs))
    B = np.repeat(b_bits, len(accs))
    acc = np.tile(accs, len(a_bits))
    r = run(scale_binary, A, B, bits(acc))
    k = -(r["ka"] + r["kb"])
    assert k.min() == -252 and k.max() == 226                              # the range the two factors must cover
    # the factors: powers of two, both fp32 normals, product 2^k
    for f in ("main", "extra"):
        v = r[f].astype(np.float64)
        assert np.all(v >= 2.0 ** -126) and np.all(v <= 2.0 ** 127)
        assert np.all(np.frexp(v)[0] == 0.5)
    assert np.array_equal(np.log2(r["main"].astype(np.float64)) + np.log2(r["extra"].astype(np.float64)), k)
    # where the whole factor is one fp32 normal, extra = 1: the epilogue's single product acc * 2^k, as it always was
    one = (k >= -126) & (k <= 127)
    assert np.all(r["extra"][one] == 1.0) and np.all(r["extra"][~one] != 1.0)
    # exact whenever the true value is an fp32 normal
    true = np.ldexp(acc.astype(np.float64), k)
    normal = (np.abs(true) >= 2.0 ** -126) & (np.abs(true) < 2.0 ** 128)
    assert normal.sum() > len(true) // 2 and (~normal).sum() > 1000
    got = r["out"].astype(np.float64)
    assert np.array_equal(got[normal], true[normal])
    # and otherwise the value an fp32 product gives: +-Inf above the range, 0 or a denormal within 2 ulp below it
    over = np.abs(true) >= 2.0 ** 128
    assert np.all(np.isinf(got[over]) & (np.sign(got[over]) == np.sign(true[over])))
    under = np.abs(true) < 2.0 ** -126
    assert np.all(np.abs(got[under] - true[under]) <= 2.0 ** -148)
