"""Shared test helpers: golden-fixture loading and error measures."""
import glob
import os

import numpy as np
import torch

from mpvae_b200 import synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
IN_KEYS = ["y", "fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma"]
GRAD_KEYS = ["fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma"]
SCALAR_KEYS = ["total_loss", "nll_loss", "nll_loss_x", "c_loss", "c_loss_x", "kl_loss"]
THRESHOLDS = [0.01, 0.02, 0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.10, 0.15, 0.20, 0.25, 0.30, 0.35, 0.40,
              0.45, 0.50, 0.55, 0.60, 0.65, 0.70, 0.75, 0.8, 0.85, 0.9, 0.95]   # train.py:22 / test.py:15


def golden_names():
    names = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    return [n for n in names if not n.startswith("metrics_")]      # metrics_cases.npz belongs to test_metrics.py


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    L, Z, B, S, D, data_seed, noise_seed = (int(v) for v in z["meta"])
    nll_coeff, c_coeff, sigma, rate = (float(v) for v in z["coeffs"])
    case = dict(name=name, L=L, Z=Z, B=B, S=S, D=D, mode=str(z["mode"]), nll_coeff=nll_coeff, c_coeff=c_coeff,
                degenerate=bool(z["degenerate"]))
    inputs = {k: z["in_" + k] for k in IN_KEYS if "in_" + k in z.files}
    if "r_sqrt_sigma" not in inputs:   # large R is regenerated from its seed
        regen = synth.loss_inputs(L, Z, B, S, seed=data_seed, sigma=sigma, label_rate=rate, latent_dim=D,
                                  with_noise=False)
        for k in IN_KEYS:
            if k in inputs:
                assert np.array_equal(regen[k], inputs[k]), k
        inputs["r_sqrt_sigma"] = regen["r_sqrt_sigma"]
    case["inputs"] = inputs
    case["noise"] = z["noise"]
    case["out"] = {k[4:]: z[k] for k in z.files if k.startswith("out_")}
    case["grad"] = {k[5:]: z[k] for k in z.files if k.startswith("grad_")}
    case["upstream"] = {k[3:]: z[k] for k in z.files if k.startswith("up_")}
    return case


def to_torch(d, device="cpu"):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(device) for k, v in d.items()}


def rel_err(a, b):
    """max |a-b| / max |b|  (tensor-max-norm relative error; 0/0 -> 0)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = np.max(np.abs(b)) if b.size else 0.0
    num = np.max(np.abs(a - b)) if b.size else 0.0
    return 0.0 if num == 0 else num / max(den, 1e-300)


def threshold_mismatches(p, q, thresholds=THRESHOLDS, tie=0.0):
    """evals.py:201-202 semantics: pred = (p >= t).  Number of differing thresholded cells whose reference
    score is further than `tie` from the threshold (tie = 0: every differing cell counts)."""
    bad = 0
    for t in thresholds:
        diff = (p >= t) != (q >= t)
        if tie > 0:
            diff &= np.abs(q.astype(np.float64) - t) > tie
        bad += int(np.sum(diff))
    return bad


def topk_mismatches(p, q, ks=(1, 3, 5), tie=2.5e-7):
    """evals.py:37: argsort descending top-k (only compared where k <= L).  A position counts as a mismatch
    only if the two implementations put labels of genuinely different score there: saturated probabilities
    (E clamps at 1 - 4.8e-7) tie to within an fp32 ulp or two and argsort's order among ties is arbitrary."""
    bad = 0
    rows = np.arange(p.shape[0])[:, None]
    for k in ks:
        if k > p.shape[1]:
            continue
        a = np.argsort(p, axis=1)[:, ::-1][:, :k]
        b = np.argsort(q, axis=1)[:, ::-1][:, :k]
        differ = a != b
        real = np.abs(q[rows, a].astype(np.float64) - q[rows, b].astype(np.float64)) > tie
        bad += int(np.sum(differ & real))
    return bad


def rel_err_l2(a, b):
    """||a-b||_2 / ||b||_2 (Frobenius): averages over rows instead of reporting the single worst cell."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = float(np.sqrt(np.sum(b * b)))
    num = float(np.sqrt(np.sum((a - b) ** 2)))
    return 0.0 if num == 0 else num / max(den, 1e-300)


def rel_err_l2_trimmed(a, b, drop=0.02):
    """rel_err_l2 with the worst `drop` fraction of ROWS (by squared error) left out of both norms.  In the dense regime
    one saturated cell -- E within an fp32 ulp of the clamp, where 1 / (1 - E) turns a 1-ulp change of noise.R^T into a
    percent-level change of that cell's gradient for ANY implementation -- can carry the whole Frobenius distance of an
    otherwise exact tensor; the trimmed norm measures everything else."""
    a = np.asarray(a, dtype=np.float64).reshape(len(a), -1)
    b = np.asarray(b, dtype=np.float64).reshape(len(b), -1)
    err = np.sum((a - b) ** 2, axis=1)
    keep = np.argsort(err)[:max(1, int(np.ceil(len(err) * (1.0 - drop))))]
    den = float(np.sqrt(np.sum(b[keep] ** 2)))
    num = float(np.sqrt(np.sum(err[keep])))
    return 0.0 if num == 0 else num / max(den, 1e-300)


# ----------------------------------------------------------------------------- element-wise bound of the tcgen05 product
def contract_c_rel(K, ksplit=False):
    """c_rel(K) of the split-precision product's element-wise error model (derivation: tests/test_contract_bound_gpu.py).
    K is the reduction length (M for the tn product)."""
    k_blocks = -(-K // 64)
    chunks = -(-k_blocks // 4)                 # TMEM chunks of kc k-blocks: kc = 4 (three-pass), 6 (two-pass)
    rounds = chunks + (14 if ksplit else 0)    # a K-sliced tail tile: up to 8 slices, each a chunk more and a fix-up add
    return 3 * 2.0 ** -22 + 8e-7 + 12 * 2.0 ** -23 + rounds * 2.0 ** -24


def contract_bound(a, b, ksplit=False):
    """For C = a . b^T (a: M x K, b: N x K, any float dtype, on the device), in fp64:
        ref   = a . b^T
        bound = c_rel(K) |a| . |b|^T + 2^-38 (max|a| ||b_j||_1 + max|b| ||a_i||_1)
    The second term is the floor of the per-tensor scale: pieces of entries below ~2^-17 of their tensor's maximum carry
    fewer than 22 bits."""
    a, b = a.double(), b.double()
    ref = a @ b.T
    aa, ab = a.abs(), b.abs()
    floor = 2.0 ** -38 * (aa.max() * ab.sum(1)[None, :] + ab.max() * aa.sum(1)[:, None])
    return ref, contract_c_rel(a.shape[1], ksplit) * (aa @ ab.T) + floor


def assert_within_contract_bound(got, a, b, ksplit=False, what="", extra=None):
    """Every element of `got` (= a . b^T computed by the engine) within contract_bound; `extra` is added to the bound
    (a caller's own rounding after the product).  Returns the worst error / bound ratio."""
    ref, bound = contract_bound(a, b, ksplit)
    if extra is not None:
        bound = bound + extra
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)                      # NaN counts as a violation
    if bool(bad.any()):
        i, j = [int(v) for v in bad.nonzero()[0]]
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.numel()} elements outside the bound; first ({i}, {j}): "
                             f"got {float(got[i, j])!r} want {float(ref[i, j])!r} err {float(err[i, j]):.3e} "
                             f"bound {float(bound[i, j]):.3e}")
    return float((err / bound.clamp_min(1e-300)).max())
