"""GPU parity tests: the CUDA path (through the C-ABI, via mpvae_b200.compute_loss) against
  (1) the committed golden vectors produced by the unmodified reference on CPU, and
  (2) the oracle restatement run on the same seeded inputs (on CPU, and on the same device).

Tolerances (north star): losses and gradients within 1e-5 relative (max-norm relative per tensor),
thresholded / ranked predictions bit-exact (evals.py:201-202, :37).  Where the reference's own fp32
summation noise exceeds that (L >= 983, see DESIGN.md "What 1e-5 means at large L") the gradient bar is
stated against the exact-sum oracle (fp32 cell arithmetic, fp64 accumulation) instead.
"""
import json
import os
import zlib

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import helpers as H

pytestmark = pytest.mark.gpu

REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report.jsonl")


def report(**kw):
    try:
        os.makedirs(os.path.dirname(REPORT), exist_ok=True)
        with open(REPORT, "a") as f:
            f.write(json.dumps(kw) + "\n")
    except OSError:
        pass


def run_cuda(inputs, noise, nll_coeff, c_coeff, mode="train", upstream=None, flags=0, need_r=True):
    from mpvae_b200.mpvae import compute_loss
    dev = torch.device("cuda:0")
    S, _, Z = noise.shape
    L = inputs["y"].shape[1]
    args = orc.make_args(L, Z, n_train_sample=S, n_test_sample=S, mode=mode, nll_coeff=nll_coeff, c_coeff=c_coeff,
                         mpvae_flags=flags)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in inputs.items() if k != "noise"}
    train = mode == "train"
    for k in H.GRAD_KEYS:
        t[k].requires_grad_(train and (need_r or k != "r_sqrt_sigma"))
    ctx = torch.enable_grad() if train else torch.no_grad()
    with ctx:
        out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                           t["r_sqrt_sigma"], args, noise=torch.from_numpy(noise).to(dev))
    grads = {}
    if train:
        obj = out[0]
        if upstream:
            obj = obj + (out[6] * torch.from_numpy(upstream["indiv_prob"]).to(dev)).sum() \
                + (out[7] * torch.from_numpy(upstream["indiv_prob_label"]).to(dev)).sum()
        obj.backward()
        grads = {k: t[k].grad.detach().cpu().numpy() for k in H.GRAD_KEYS if t[k].grad is not None}
    torch.cuda.synchronize()
    outs = {k: o.detach().cpu().numpy() for k, o in zip(H.SCALAR_KEYS + ["indiv_prob", "indiv_prob_label"], out)}
    return outs, grads


def run_oracle(inputs, noise, nll_coeff, c_coeff, mode="train", upstream=None, device="cpu", **kw):
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(device) for k, v in inputs.items() if k != "noise"}
    nz = torch.from_numpy(noise).to(device)
    if mode == "train":
        up = None
        if upstream:
            up = {"total_loss": torch.tensor(1.0, device=device)}
            up.update({k: torch.from_numpy(v).to(device) for k, v in upstream.items()})
        terms, grads = orc.probit_elbo_with_grads(t, nz, nll_coeff, c_coeff, upstream=up, **kw)
        grads = {k: g.detach().cpu().numpy() for k, g in grads.items()}
    else:
        with torch.no_grad():
            terms = orc.probit_elbo(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"],
                                    t["fx_logvar"], t["r_sqrt_sigma"], nz, nll_coeff, c_coeff, **kw)
        grads = {}
    outs = {k: o.detach().cpu().numpy() for k, o in zip(H.SCALAR_KEYS + ["indiv_prob", "indiv_prob_label"], terms)}
    return outs, grads


def measure(got_o, got_g, ref_o, ref_g, nan_ok=False):
    errs = {}
    for k in H.SCALAR_KEYS:
        errs[k] = H.rel_err(got_o[k], ref_o[k])
    for k in ("indiv_prob", "indiv_prob_label"):
        errs[k + "_abs"] = float(np.max(np.abs(got_o[k].astype(np.float64) - ref_o[k]))) if ref_o[k].size else 0.0
    errs["threshold_flips"] = H.threshold_mismatches(got_o["indiv_prob"], ref_o["indiv_prob"]) \
        + H.threshold_mismatches(got_o["indiv_prob_label"], ref_o["indiv_prob_label"])
    errs["topk_flips"] = H.topk_mismatches(got_o["indiv_prob"], ref_o["indiv_prob"])
    for k, g in ref_g.items():
        if k not in got_g:
            continue
        if nan_ok:
            errs["g_" + k + "_nanpattern"] = bool(np.array_equal(np.isnan(got_g[k]), np.isnan(g)))
            errs["g_" + k] = H.rel_err(np.nan_to_num(got_g[k]), np.nan_to_num(g))
        else:
            errs["g_" + k] = H.rel_err(got_g[k], g)
    return errs


def compare(tag, got_o, got_g, ref_o, ref_g, tol_loss=1e-5, tol_grad=1e-5, tol_grad_r=None, nan_ok=False, floor=None):
    """Assert the north-star bars.  `floor` (optional, per gradient key) is the distance between the reference's
    own CUDA and CPU runs on these inputs: against a CPU-generated fixture the kernel is held to
    max(tol, 2 * floor), because 1-ulp differences between libm and libdevice erff are amplified by
    1/(1-E) in saturated cells no matter who computes them (SURVEY section 7, hard part 1)."""
    errs = measure(got_o, got_g, ref_o, ref_g, nan_ok)
    rec = {k: (v if isinstance(v, (bool, int)) else float(v)) for k, v in errs.items()}
    if floor:
        rec.update({"floor_" + k: float(v) for k, v in floor.items()})
    report(tag=tag, **rec)
    for k in H.SCALAR_KEYS:
        tol = max(tol_loss, 2.0 * floor.get(k, 0.0)) if floor else tol_loss
        assert errs[k] <= tol, (tag, k, errs[k], tol)
    # |mean_s E| differs from torch's reduction order by a few fp32 ulps; what must be exact is the decision
    assert errs["indiv_prob_abs"] <= 5e-7 and errs["indiv_prob_label_abs"] <= 5e-7, (tag, errs)
    assert errs["threshold_flips"] == 0, (tag, "thresholded predictions differ", errs["threshold_flips"])
    assert errs["topk_flips"] == 0, (tag, "top-k ranking differs")
    for k in ref_g:
        if k not in got_g:
            continue
        tol = tol_grad_r if (k == "r_sqrt_sigma" and tol_grad_r is not None) else tol_grad
        if floor and k in floor:
            tol = max(tol, 2.0 * floor[k])
        assert errs["g_" + k] <= tol, (tag, k, errs["g_" + k], tol)
        if nan_ok:
            assert errs["g_" + k + "_nanpattern"], (tag, k, "NaN pattern differs")
    return errs


def grad_floor(dev_g, cpu_g, nan_ok=False, dev_o=None, cpu_o=None):
    out = {}
    if dev_o is not None:
        for k in H.SCALAR_KEYS:
            out[k] = H.rel_err(dev_o[k], cpu_o[k])
    for k, g in cpu_g.items():
        if k in dev_g:
            out[k] = H.rel_err(np.nan_to_num(dev_g[k]), np.nan_to_num(g)) if nan_ok else H.rel_err(dev_g[k], g)
    return out


@pytest.mark.parametrize("name", H.golden_names())
def test_golden_vectors(name):
    """Fixtures = the unmodified reference run on CPU.  Forward at 1e-5, decisions exact; gradients at 1e-5 or
    twice the reference's own CUDA-vs-CPU distance on the same inputs, whichever is larger."""
    case = H.load_golden(name)
    up = case["upstream"] or None
    got_o, got_g = run_cuda(case["inputs"], case["noise"], case["nll_coeff"], case["c_coeff"], mode=case["mode"],
                            upstream=up)
    ref_g = {k: v for k, v in case["grad"].items() if not k.startswith("r_digest")}
    if case["mode"] == "train":
        assert got_g["r_sqrt_sigma"].dtype == np.float64      # the Parameter is fp64 (SURVEY 8a-2)
    ranking = "pairwise" if case["L"] <= 1000 else "factorised"
    dev_o, dev_g = run_oracle(case["inputs"], case["noise"], case["nll_coeff"], case["c_coeff"], mode=case["mode"],
                              upstream=up, device="cuda:0", ranking=ranking)
    floor = grad_floor(dev_g, ref_g, case["degenerate"], dev_o, case["out"])
    compare("golden/" + name, got_o, got_g, case["out"], ref_g, nan_ok=case["degenerate"], floor=floor,
            tol_loss=2e-5 if name == "mirflickr_tails" else 1e-5)
    if "r_digest_sub" in case["grad"]:
        g, d = got_g["r_sqrt_sigma"], dev_g["r_sqrt_sigma"]
        tol = max(1e-5, 2 * H.rel_err(d[::29, ::31], case["grad"]["r_digest_sub"]))
        assert H.rel_err(g[::29, ::31], case["grad"]["r_digest_sub"]) <= tol
        tol = max(1e-5, 2 * H.rel_err(d.sum(1), case["grad"]["r_digest_rowsum"]))
        assert H.rel_err(g.sum(1), case["grad"]["r_digest_rowsum"]) <= tol


SHAPES = {
    # name: (L, Z, B, S, mode, sigma, rate)         BASELINE.json configs at full size where the oracle fits
    "C1_mirflickr": (38, 38, 128, 10, "train", 1.0, 0.1),
    "C2_yeast": (14, 14, 128, 10, "train", 1.0, 0.1),
    "C3_nuswide_test": (81, 81, 128, 100, "test", 1.0, 0.1),
    "C1_sigma05": (38, 38, 128, 10, "train", 0.5, 0.1),
    "C1_sigma3_tails": (38, 38, 128, 10, "train", 3.0, 0.1),
    "lowrank_L81_Z10": (81, 10, 128, 10, "train", 1.0, 0.1),
    "ragged_B77": (38, 38, 77, 10, "train", 1.0, 0.1),
    "S3_L130_Z5": (130, 5, 33, 3, "train", 1.0, 0.1),
    "S100_train": (38, 38, 32, 100, "train", 1.0, 0.1),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_full_size_against_oracle(name):
    """The reference's own PyTorch path on the same device (oracle restatement on cuda: same ATen kernels, same
    libdevice erff/logf/expf) is the strict 1e-5 bar; the CPU run of it is held to the cross-device floor."""
    from mpvae_b200 import synth
    L, Z, B, S, mode, sigma, rate = SHAPES[name]
    inp = synth.loss_inputs(L, Z, B, S, seed=zlib.crc32(name.encode()) % 1000 + 1, sigma=sigma, label_rate=rate)
    noise = inp.pop("noise")
    got_o, got_g = run_cuda(inp, noise, 0.5, 10.0, mode=mode)
    dev_o, dev_g = run_oracle(inp, noise, 0.5, 10.0, mode=mode, device="cuda:0")
    compare("oracle_cuda/" + name, got_o, got_g, dev_o, dev_g, tol_loss=2e-5 if "tails" in name else 1e-5)
    ref_o, ref_g = run_oracle(inp, noise, 0.5, 10.0, mode=mode, device="cpu")
    compare("oracle_cpu/" + name, got_o, got_g, ref_o, ref_g, floor=grad_floor(dev_g, ref_g, False, dev_o, ref_o),
            tol_loss=2e-5 if "tails" in name else 1e-5)


@pytest.mark.parametrize("name,L,Z,B", [("delicious", 983, 983, 16), ("delicious_z10", 983, 10, 16),
                                        ("eurlex_z10", 3993, 10, 4)])
def test_large_label_sets_against_exact_sum_oracle(name, L, Z, B):
    """At L >= 983 the 1e-5 bar is checked against the oracle with fp64 accumulation (same fp32 cell
    arithmetic, exact sums); the plain fp32 oracle is reported next to it to show its own order noise."""
    from mpvae_b200 import synth
    S = 10
    inp = synth.loss_inputs(L, Z, B, S, seed=31, sigma=1.0, label_rate=20.0 / L)
    noise = inp.pop("noise")
    from mpvae_b200 import _lib
    # CUDA-core contraction: same fp32 FMA chain as the reference's SGEMM, so the exact-sum oracle is the 1e-5 bar
    got_o, got_g = run_cuda(inp, noise, 0.5, 10.0, flags=_lib.FLAG_CONTRACT_FMA)
    ex_o, ex_g = run_oracle(inp, noise, 0.5, 10.0, device="cuda:0", ranking="factorised", accum=torch.float64)
    errs = compare("exact_sum/" + name, got_o, got_g, ex_o, ex_g, tol_grad=1e-5, tol_grad_r=2e-5)
    f32_o, f32_g = run_oracle(inp, noise, 0.5, 10.0, device="cuda:0", ranking="factorised")
    noise_floor = {k: H.rel_err(f32_g[k], ex_g[k]) for k in ex_g}
    report(tag="fp32_oracle_vs_exact_sum/" + name, **{k: float(v) for k, v in noise_floor.items()})
    assert errs["g_fe_out"] <= max(1e-5, noise_floor["fe_out"])


@pytest.mark.parametrize("name,L,Z,B", [("delicious", 983, 983, 16), ("delicious_b128", 983, 983, 128),
                                        ("eurlex_b16", 3993, 3993, 16)])
def test_tensor_engine_is_as_accurate_as_the_reference(name, L, Z, B):
    """Dense regime (Z >= 128): noise.R^T runs as a split-precision product on tcgen05, whose rounding differs from an fp32 SGEMM's
    (it is ~2x closer to the exact product).  At these sizes a 1e-6 perturbation of x moves softmax_s(lp) -- and
    with it every gradient -- by ~sqrt(L) * 1e-6 * |dll/dx| ~ 1e-4, for ANY implementation including the
    reference's own cuBLAS path.  So the bar is: forward terms within 1e-5 of the reference path, decisions equal
    away from ties, and gradients at least as close to the exact-contraction truth (fp64 product, exact sums, fp32
    cell arithmetic) as the reference's own fp32 path is."""
    from mpvae_b200 import _lib, synth
    S = 10
    inp = synth.loss_inputs(L, Z, B, S, seed=32, sigma=1.0, label_rate=20.0 / L)
    noise = inp.pop("noise")
    got_o, got_g = run_cuda(inp, noise, 0.5, 10.0, flags=_lib.FLAG_CONTRACT_TENSOR)
    ref_o, ref_g = run_oracle(inp, noise, 0.5, 10.0, device="cuda:0", ranking="factorised")
    tru_o, tru_g = run_oracle(inp, noise, 0.5, 10.0, device="cuda:0", ranking="factorised", accum=torch.float64,
                              contract=torch.float64)
    rec = {}
    for k in H.SCALAR_KEYS:
        rec[k] = H.rel_err(got_o[k], ref_o[k])
        assert rec[k] <= 1e-5, (k, rec[k])
    dp = float(np.max(np.abs(got_o["indiv_prob"].astype(np.float64) - ref_o["indiv_prob"])))
    rec["indiv_prob_abs"] = dp
    assert dp <= 5e-6
    # decisions may only differ where the reference score sits within the two paths' distance of a threshold
    assert H.threshold_mismatches(got_o["indiv_prob"], ref_o["indiv_prob"], tie=2 * dp + 1e-7) == 0
    rec["threshold_ties"] = H.threshold_mismatches(got_o["indiv_prob"], ref_o["indiv_prob"])
    # Frobenius-relative distance to the truth (the max-norm is decided by one saturated cell of one row and
    # fluctuates by 10x between two equally accurate implementations; it is recorded, and capped at 2e-3)
    for k in H.GRAD_KEYS:
        mine, theirs = H.rel_err_l2(got_g[k], tru_g[k]), H.rel_err_l2(ref_g[k], tru_g[k])
        rec["g_" + k], rec["ref_" + k] = mine, theirs
        rec["gmax_" + k], rec["refmax_" + k] = H.rel_err(got_g[k], tru_g[k]), H.rel_err(ref_g[k], tru_g[k])
    report(tag="tensor_vs_truth/" + name, **{k: float(v) for k, v in rec.items()})
    for k in H.GRAD_KEYS:
        assert rec["g_" + k] <= max(1e-5, 2.0 * rec["ref_" + k]), (k, rec["g_" + k], rec["ref_" + k])
        assert rec["gmax_" + k] <= 2e-3, (k, rec["gmax_" + k])


@pytest.mark.parametrize("L,Z,B", [(256, 253, 64), (256, 254, 64), (255, 255, 64), (130, 256, 70), (983, 983, 128)])
def test_library_noise_in_the_dense_regime(L, Z, B):
    """With `noise=None` the library draws Philox normals on the fp16 grid straight into ONE operand plane and runs the
    two-pass products (contract_tc.cu EX = 1 / 2).  The same numbers come out of `philox_normal`; fed back as an
    external tensor they take the split + three-pass route.  Both routes -- and the reference's torch path on the
    same noise -- must agree: this pins the plane writer (all four destination alignments: Z mod 4 = 1, 2, 3, 0), the
    exact-operand kernels and the gxs planes the row backward writes with its a-priori scale."""
    from mpvae_b200 import synth
    from mpvae_b200.mpvae import compute_loss
    from mpvae_b200.probit import philox_normal
    S = 10
    inp = synth.loss_inputs(L, Z, B, S, seed=77, sigma=1.0, label_rate=max(0.05, 20.0 / L), with_noise=False)
    dev = torch.device("cuda:0")

    def run(external):
        args = orc.make_args(L, Z, n_train_sample=S, noise_seed=909, noise_offset=3)
        t = {k: torch.from_numpy(v).to(dev).requires_grad_(k != "y") for k, v in inp.items()}
        kw = {"noise": philox_normal(S, B, Z, seed=909, offset=3, device=dev)} if external else {}
        out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                           t["r_sqrt_sigma"], args, **kw)
        out[0].backward()
        return ([o.detach().cpu().numpy() for o in out], {k: t[k].grad.cpu().numpy() for k in H.GRAD_KEYS})

    lib_o, lib_g = run(False)
    ext_o, ext_g = run(True)
    noise = philox_normal(S, B, Z, seed=909, offset=3, device=dev)
    assert torch.equal(noise, noise.half().float())                       # on the fp16 grid
    nz = noise.cpu().numpy()
    ref_o, ref_g = run_oracle(inp, nz, 0.5, 10.0, device="cuda:0", ranking="factorised")
    tru_o, tru_g = run_oracle(inp, nz, 0.5, 10.0, device="cuda:0", ranking="factorised", accum=torch.float64,
                              contract=torch.float64)
    rec = {}
    for i, k in enumerate(H.SCALAR_KEYS):
        rec["two_vs_three_" + k] = H.rel_err(lib_o[i], ext_o[i])
        rec[k] = H.rel_err(lib_o[i], ref_o[k])
        assert rec["two_vs_three_" + k] <= 2e-6, (k, "two-pass vs three-pass")
        assert rec[k] <= 1e-5, (k, "vs the torch path")
    assert float(np.max(np.abs(lib_o[6] - ext_o[6]))) <= 2e-6
    assert float(np.max(np.abs(lib_o[6] - ref_o["indiv_prob"]))) <= 5e-6
    # gradients: the same rule as test_tensor_engine_is_as_accurate_as_the_reference -- at least as close to the
    # exact-contraction truth (Frobenius, x2 slack) as the reference's own fp32 torch path, for BOTH routes.  A single
    # saturated cell can carry the whole-tensor norm (helpers.rel_err_l2_trimmed): the rule must hold on the whole
    # tensor or, with the worst 2 % of rows set aside on both sides, on the rest -- and the whole tensor stays under 1e-4.
    bad = []
    for k in H.GRAD_KEYS:
        theirs, theirs_t = H.rel_err_l2(ref_g[k], tru_g[k]), H.rel_err_l2_trimmed(ref_g[k], tru_g[k])
        for route, g in (("two_pass", lib_g), ("three_pass", ext_g)):
            mine, mine_t = H.rel_err_l2(g[k], tru_g[k]), H.rel_err_l2_trimmed(g[k], tru_g[k])
            rec[f"g_{route}_{k}"], rec[f"gtrim_{route}_{k}"] = mine, mine_t
            rec[f"gmax_{route}_{k}"] = H.rel_err(g[k], tru_g[k])
            ok = mine <= max(1e-5, 2.0 * theirs) or (mine_t <= max(1e-5, 2.0 * theirs_t) and mine <= 1e-4)
            if not ok:
                bad.append((route, k, mine, theirs, mine_t, theirs_t))
        rec["ref_" + k] = theirs
        rec["refmax_" + k] = H.rel_err(ref_g[k], tru_g[k])
        rec["two_vs_three_g_" + k] = H.rel_err_l2(lib_g[k], ext_g[k])
    report(tag=f"library_noise_dense/L{L}_Z{Z}_B{B}", **{k: float(v) for k, v in rec.items()})
    assert not bad, bad


@pytest.mark.parametrize("S,B,L,Z,external,weighted", [
    (10, 128, 983, 983, False, False), (10, 70, 300, 256, False, False), (3, 77, 130, 256, True, False),
    (7, 33, 513, 130, False, False), (100, 12, 300, 128, True, False), (1, 300, 256, 256, False, False),
    (256, 5, 257, 128, False, False), (10, 1024, 3993, 3993, False, False), (10, 70, 300, 256, False, True)])
def test_removed_fused_flags_give_the_default_bits(S, B, L, Z, external, weighted):
    """MPVAE_FLAG_FUSED_FORWARD and MPVAE_FLAG_FUSED_EXCHANGE selected paths that were measured slower and removed; the
    library accepts and ignores them.  Dense regime: all 8 outputs and every gradient bit for bit as with flags = 0, with a
    label mask, row weights and label weights too (weighted).  Shapes: S from 1 to 256, ragged last tiles, and bench.py's
    headline configuration."""
    from mpvae_b200 import _lib, synth
    from mpvae_b200.mpvae import compute_loss
    inp = synth.loss_inputs(L, Z, B, S, seed=S + B, sigma=1.0, label_rate=max(0.05, 20.0 / L), with_noise=external)
    dev = torch.device("cuda:0")
    noise = torch.from_numpy(inp.pop("noise")).to(dev) if external else None
    kw = {"noise": noise} if external else {}
    if weighted:
        g = torch.Generator().manual_seed(L)
        kw.update(label_mask=(torch.rand(B, L, generator=g) < 0.6).to(dev), row_weight=(torch.rand(B, generator=g) * 2.0).to(dev),
                  pos_weight=(torch.rand(L, generator=g) * 3.0).to(dev), neg_weight=(torch.rand(L, generator=g) + 0.5).to(dev))

    def run(flags):
        args = orc.make_args(L, Z, n_train_sample=S, noise_seed=31337, noise_offset=9, mpvae_flags=flags | _lib.FLAG_CONTRACT_TENSOR)
        t = {k: torch.from_numpy(v).to(dev).requires_grad_(k != "y") for k, v in inp.items()}
        out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                           t["r_sqrt_sigma"], args, **kw)
        out[0].backward()
        torch.cuda.synchronize()
        return [o.detach().cpu().numpy() for o in out], {k: t[k].grad.cpu().numpy() for k in H.GRAD_KEYS}

    flagged_o, flagged_g = run(_lib.FLAG_FUSED_FORWARD | _lib.FLAG_FUSED_EXCHANGE)
    plain_o, plain_g = run(0)
    for a, b in zip(flagged_o, plain_o):
        np.testing.assert_array_equal(a, b)
    for k in H.GRAD_KEYS:
        np.testing.assert_array_equal(flagged_g[k], plain_g[k])


@pytest.mark.parametrize("S,B,L,Z,external,mode", [(10, 128, 38, 38, True, "train"), (10, 128, 38, 38, False, "train"),
                                                   (10, 128, 14, 14, False, "train"), (100, 128, 81, 81, False, "test"),
                                                   (3, 33, 128, 5, True, "train"), (7, 77, 81, 81, False, "train"),
                                                   (1, 5, 2, 1, True, "train"), (100, 32, 38, 38, False, "train"),
                                                   (11, 300, 50, 127, False, "train")])
def test_small_regime_kernel_equals_the_general_path(S, B, L, Z, external, mode):
    """Label / rank sets that fit an SM (C1-C3 of BASELINE.json) run as ONE fused launch per direction
    (probit_small_fwd_kernel: R staged by a TMA bulk copy, Philox in registers, warp-FMA contraction, row math, tail).
    MPVAE_FLAG_CONTRACT_FMA forces the general path (Philox kernel, CUDA-core GEMM, tiled forward, finalize).  Same FMA
    chain, same cell arithmetic, same sample order: every forward output must be BIT-equal; gradients differ only in
    summation order (samples for the logit gradients, batch rows for g_R)."""
    from mpvae_b200 import _lib, synth
    from mpvae_b200.mpvae import compute_loss
    inp = synth.loss_inputs(L, Z, B, S, seed=7 * S + B, sigma=1.0, label_rate=0.1, with_noise=external)
    dev = torch.device("cuda:0")
    noise = torch.from_numpy(inp.pop("noise")).to(dev) if external else None
    train = mode == "train"

    def run(flags):
        args = orc.make_args(L, Z, n_train_sample=S, n_test_sample=S, mode=mode, noise_seed=4711, noise_offset=2, mpvae_flags=flags)
        t = {k: torch.from_numpy(v).to(dev).requires_grad_(train and k != "y") for k, v in inp.items()}
        launches0 = _lib.launch_count()
        with torch.enable_grad() if train else torch.no_grad():
            out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                               t["r_sqrt_sigma"], args, **({"noise": noise} if external else {}))
            if train:
                out[0].backward()
        torch.cuda.synchronize()
        n_launch = _lib.launch_count() - launches0
        return ([o.detach().cpu().numpy() for o in out], {k: t[k].grad.cpu().numpy() for k in H.GRAD_KEYS} if train else {}, n_launch)

    small_o, small_g, n_small = run(0)
    gen_o, gen_g, n_gen = run(_lib.FLAG_CONTRACT_FMA)
    assert n_small == (3 if train else 1), n_small           # forward 1, backward 2 (rows + the ordered g_R sum)
    assert n_gen > n_small
    for a, b in zip(small_o, gen_o):
        np.testing.assert_array_equal(a, b)
    for k in small_g:
        # logit gradients: the same cells summed over samples in a different (fixed) order; g_R: rows summed in order
        assert H.rel_err(small_g[k], gen_g[k]) <= (2e-6 if k == "r_sqrt_sigma" else 5e-7), (k, H.rel_err(small_g[k], gen_g[k]))
    again_o, again_g, _ = run(0)
    for a, b in zip(small_o, again_o):
        np.testing.assert_array_equal(a, b)
    for k in small_g:
        np.testing.assert_array_equal(small_g[k], again_g[k])


def test_headline_configuration_rows_against_the_oracle():
    """bench.py's default workload -- eurlex-shaped S10 B1024 L3993 Z3993, the library's own Philox noise, two-pass tensor
    product and the separate row forward -- has no O(L^2)-sized oracle run.  It is tied to the oracle through a 16-row
    window: (1) the library on rows [r0, r0 + 16) alone, drawing the SAME noise rows (global-row Philox keying), gives
    bit-equal predictions and, rescaled by B / 16, the same logit gradients as the full-batch run; (2) that window agrees
    with the reference's torch path (oracle on the same device, fed `philox_normal`) at the north-star bars: forward
    1e-5, decisions equal away from ties, gradients at least as close to the exact-contraction truth as the
    reference's own fp32 path."""
    from mpvae_b200 import synth
    from mpvae_b200.mpvae import compute_loss
    from mpvae_b200.probit import philox_normal
    L = Z = 3993
    B, S, r0, nw = 1024, 10, 512 - 8, 16
    inp = synth.loss_inputs(L, Z, B, S, seed=3, label_rate=20.0 / L, with_noise=False)
    dev = torch.device("cuda:0")

    def run(lo, hi):
        args = orc.make_args(L, Z, n_train_sample=S, noise_seed=777, noise_offset=5, dp_global_batch=B, dp_row0=lo)
        t = {k: torch.from_numpy(v if k == "r_sqrt_sigma" else v[lo:hi]).to(dev).requires_grad_(k != "y") for k, v in inp.items()}
        out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                           t["r_sqrt_sigma"], args)
        out[0].backward()
        return [o.detach().cpu().numpy() for o in out], {k: t[k].grad.cpu().numpy() for k in H.GRAD_KEYS}

    full_o, full_g = run(0, B)
    win_o, win_g = run(r0, r0 + nw)
    np.testing.assert_array_equal(full_o[6][r0:r0 + nw], win_o[6])
    np.testing.assert_array_equal(full_o[7][r0:r0 + nw], win_o[7])
    rec = {}
    for k in ("fe_out", "fx_out", "fe_mu", "fx_logvar"):
        rec["window_g_" + k] = H.rel_err(full_g[k][r0:r0 + nw] * (B / nw), win_g[k])
        assert rec["window_g_" + k] <= 2e-6, (k, rec)
    noise = philox_normal(S, nw, Z, seed=777, offset=5, device=dev, global_batch=B, row0=r0).cpu().numpy()
    sub = {k: (v if k == "r_sqrt_sigma" else v[r0:r0 + nw]) for k, v in inp.items()}
    ref_o, ref_g = run_oracle(sub, noise, 0.5, 10.0, device="cuda:0", ranking="factorised")
    tru_o, tru_g = run_oracle(sub, noise, 0.5, 10.0, device="cuda:0", ranking="factorised", accum=torch.float64,
                              contract=torch.float64)
    for i, k in enumerate(H.SCALAR_KEYS):
        rec[k] = H.rel_err(win_o[i], ref_o[k])
        assert rec[k] <= 1e-5, (k, rec[k])
    dp = float(np.max(np.abs(win_o[6].astype(np.float64) - ref_o["indiv_prob"])))
    rec["indiv_prob_abs"] = dp
    assert dp <= 5e-6
    assert H.threshold_mismatches(win_o[6], ref_o["indiv_prob"], tie=2 * dp + 1e-7) == 0
    for k in H.GRAD_KEYS:
        mine, theirs = H.rel_err_l2(win_g[k], tru_g[k]), H.rel_err_l2(ref_g[k], tru_g[k])
        rec["g_" + k], rec["ref_" + k] = mine, theirs
        assert mine <= max(1e-5, 2.0 * theirs), (k, mine, theirs)
    report(tag="headline_eurlex_B1024_philox_window16", **{k: float(v) for k, v in rec.items()})


def test_stable_cdf_flag_is_closer_to_the_exact_formula():
    """MPVAE_FLAG_STABLE_CDF (opt-in; north_star's "numerically stable erfc form"): Phi and 1 - Phi from erfc(|x|/sqrt 2).
    The reference's own fp32 form 0.5 (1 + erf) cancels in the tails; evaluated in fp64 the same formula is the truth
    both modes are measured against.  On a tail-heavy case (logit sigma 3) the stable mode must sit much closer to it
    than the faithful mode does -- which is also why the flag is off by default: parity is with the reference."""
    from mpvae_b200 import _lib, synth
    L, Z, B, S = 38, 38, 64, 10
    inp = synth.loss_inputs(L, Z, B, S, seed=8, sigma=3.0)
    noise = inp.pop("noise")
    faithful_o, faithful_g = run_cuda(inp, noise, 0.5, 10.0)
    stable_o, stable_g = run_cuda(inp, noise, 0.5, 10.0, flags=_lib.FLAG_STABLE_CDF)
    truth_o, truth_g = run_oracle(inp, noise, 0.5, 10.0, device="cuda:0", dtype=torch.float64)
    rec = {}
    for k in ("nll_loss", "nll_loss_x", "total_loss"):
        rec["faithful_" + k], rec["stable_" + k] = H.rel_err(faithful_o[k], truth_o[k]), H.rel_err(stable_o[k], truth_o[k])
        assert rec["stable_" + k] <= 2e-6, (k, rec)
    for k in ("fe_out", "fx_out", "r_sqrt_sigma"):
        rec["faithful_g_" + k] = H.rel_err_l2(faithful_g[k], truth_g[k])
        rec["stable_g_" + k] = H.rel_err_l2(stable_g[k], truth_g[k])
        assert rec["stable_g_" + k] <= 5e-6, (k, rec)
        assert rec["stable_g_" + k] <= 0.2 * rec["faithful_g_" + k], (k, rec)
    report(tag="stable_cdf_vs_fp64", **{k: float(v) for k, v in rec.items()})
    assert float(np.max(np.abs(stable_o["indiv_prob"] - truth_o["indiv_prob"]))) <= 1e-6


def test_upstream_on_every_output():
    """Cotangents on all 8 outputs at once (autograd contract, SURVEY 8b)."""
    from mpvae_b200 import synth
    from mpvae_b200.mpvae import compute_loss
    L, Z, B, S = 38, 10, 24, 10
    inp = synth.loss_inputs(L, Z, B, S, seed=5)
    noise = inp.pop("noise")
    rng = np.random.RandomState(3)
    w = rng.standard_normal(6).astype(np.float32)
    up_p = rng.standard_normal((B, L)).astype(np.float32)
    up_l = rng.standard_normal((B, L)).astype(np.float32)
    dev = torch.device("cuda:0")
    args = orc.make_args(L, Z, n_train_sample=S)

    def objective(fn, device, **kw):
        t = {k: torch.from_numpy(v).to(device).requires_grad_(k != "y") for k, v in inp.items()}
        out = fn(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                 t["r_sqrt_sigma"], args, noise=torch.from_numpy(noise).to(device), **kw)
        obj = sum(float(w[i]) * out[i] for i in range(6)) + (out[6] * torch.from_numpy(up_p).to(device)).sum() \
            + (out[7] * torch.from_numpy(up_l).to(device)).sum()
        obj.backward()
        return {k: t[k].grad.cpu().numpy() for k in H.GRAD_KEYS}

    got = objective(compute_loss, dev)
    ref = objective(orc.compute_loss, "cpu")
    for k in H.GRAD_KEYS:
        assert H.rel_err(got[k], ref[k]) <= 1e-5, (k, H.rel_err(got[k], ref[k]))


def test_sanitize_flag_zeroes_degenerate_ranking_gradient():
    from mpvae_b200 import _lib
    case = H.load_golden("degenerate_rows")
    got_o, got_g = run_cuda(case["inputs"], case["noise"], case["nll_coeff"], case["c_coeff"],
                            flags=_lib.FLAG_SANITIZE_DEGENERATE)
    for k in H.SCALAR_KEYS:
        assert H.rel_err(got_o[k], case["out"][k]) <= 1e-5
    for k, g in got_g.items():
        assert np.isfinite(g).all(), k
    good = [0, 2, 3, 5]
    assert H.rel_err(got_g["fe_out"][good], case["grad"]["fe_out"][good]) <= 1e-5


def test_frozen_r_gets_no_gradient():
    case = H.load_golden("yeast_b16")
    got_o, got_g = run_cuda(case["inputs"], case["noise"], case["nll_coeff"], case["c_coeff"], need_r=False)
    assert "r_sqrt_sigma" not in got_g
    assert H.rel_err(got_g["fe_out"], case["grad"]["fe_out"]) <= 1e-5


def test_empty_batch_gives_nan_means():
    """train.py:102 / fairsoft_train.py:45 run int(N/bs)+1 steps: B == 0 reaches the loss when bs | N."""
    from mpvae_b200.mpvae import compute_loss
    dev = torch.device("cuda:0")
    L, Z, D = 14, 14, 50
    args = orc.make_args(L, Z)
    e = lambda *s: torch.empty(*s, device=dev)
    out = compute_loss(e(0, L), e(0, L), e(0, D), e(0, D), e(0, L), e(0, D), e(0, D),
                       torch.zeros(L, Z, dtype=torch.float64, device=dev), args)
    assert all(torch.isnan(o).item() for o in out[:6])
    assert out[6].shape == (0, L) and out[7].shape == (0, L)


def test_rejects_cpu_tensors_loudly():
    from mpvae_b200.mpvae import compute_loss
    case = H.load_golden("yeast_b16")
    t = H.to_torch(case["inputs"])
    args = orc.make_args(case["L"], case["Z"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                     t["r_sqrt_sigma"], args)


def test_deterministic_and_reusable():
    """Same inputs twice -> identical bits (fixed-order reductions everywhere); in-place add on the returned
    total_loss is allowed (fairsoft_train.py:136 does `total_loss += fairloss`)."""
    case = H.load_golden("mirflickr_b16")
    a_o, a_g = run_cuda(case["inputs"], case["noise"], case["nll_coeff"], case["c_coeff"])
    b_o, b_g = run_cuda(case["inputs"], case["noise"], case["nll_coeff"], case["c_coeff"])
    for k in a_o:
        np.testing.assert_array_equal(a_o[k], b_o[k])
    for k in a_g:
        np.testing.assert_array_equal(a_g[k], b_g[k])
    from mpvae_b200.mpvae import compute_loss
    dev = torch.device("cuda:0")
    t = {k: torch.from_numpy(v).to(dev).requires_grad_(k != "y") for k, v in case["inputs"].items()}
    args = orc.make_args(case["L"], case["Z"], n_train_sample=case["S"])
    out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                       t["r_sqrt_sigma"], args, noise=torch.from_numpy(case["noise"]).to(dev))
    total = out[0]
    total += 3.0 * out[6].mean()
    total.backward()
    assert torch.isfinite(t["fx_out"].grad).all()


def test_inference_with_many_samples():
    """main.py:33 defaults n_test_sample to 10000: the sample axis is streamed, not held; checked at S = 2000."""
    from mpvae_b200 import synth
    L, Z, B, S = 38, 38, 12, 2000
    inp = synth.loss_inputs(L, Z, B, S, seed=77, sigma=1.0)
    noise = inp.pop("noise")
    got_o, _ = run_cuda(inp, noise, 0.5, 10.0, mode="test")
    dev_o, _ = run_oracle(inp, noise, 0.5, 10.0, mode="test", device="cuda:0")
    for k in H.SCALAR_KEYS:
        assert H.rel_err(got_o[k], dev_o[k]) <= 1e-5, (k, H.rel_err(got_o[k], dev_o[k]))
    assert H.threshold_mismatches(got_o["indiv_prob"], dev_o["indiv_prob"], tie=2.5e-7) == 0
    assert float(np.max(np.abs(got_o["indiv_prob"] - dev_o["indiv_prob"]))) <= 2e-6   # S = 2000 fp32 mean


def test_integration_stub_runs():
    """INTEGRATION.md section 2: the condensed ctypes binding (struct without the peer_* fields) drives the library's
    forward and agrees with the maintained binding on the same noise."""
    from tests.test_lib_cpu import _integration_stub_source
    from mpvae_b200.mpvae import compute_loss
    ns = {}
    exec(_integration_stub_source(), ns)
    case = H.load_golden("mirflickr_b16")
    dev = torch.device("cuda:0")
    t = {k: torch.from_numpy(v).to(dev) for k, v in case["inputs"].items()}
    noise = torch.from_numpy(case["noise"]).to(dev)
    args = orc.make_args(case["L"], case["Z"], n_train_sample=case["S"])
    with torch.no_grad():
        got = ns["_ProbitELBO"].apply(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                                      t["r_sqrt_sigma"].float(), noise, args.nll_coeff, args.c_coeff)
        want = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                            t["r_sqrt_sigma"], args, noise=noise)
    torch.cuda.synchronize()
    for a, b in zip(got, want):
        assert torch.equal(a, b)


@pytest.mark.parametrize("S,B,L,Z", [(10, 16, 38, 38), (10, 33, 983, 10), (7, 33, 513, 130), (10, 128, 983, 983), (3, 77, 130, 256)])
def test_poisoned_scratch_does_not_leak(S, B, L, Z, monkeypatch):
    """compute-sanitizer (initcheck) is closed on this pool.  Stand-in: with MPVAE_POISON_WORKSPACE=1 the host wrapper fills
    the scratch block and every output buffer with 0xFF bytes (NaN in every float format, huge as a counter) before the
    calls; the three regimes (small, CUDA-core, tensor engine -- incl. ragged tiles and operand-plane padding) must
    return exactly what they return on fresh memory, i.e. nothing is read before the library wrote it."""
    from mpvae_b200 import synth
    from mpvae_b200.mpvae import compute_loss
    inp = synth.loss_inputs(L, Z, B, S, seed=S + L, sigma=1.0, label_rate=max(0.05, 20.0 / L), with_noise=False)
    dev = torch.device("cuda:0")

    def run():
        args = orc.make_args(L, Z, n_train_sample=S, noise_seed=99, noise_offset=4)
        t = {k: torch.from_numpy(v).to(dev).requires_grad_(k != "y") for k, v in inp.items()}
        out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                           t["r_sqrt_sigma"], args)
        out[0].backward()
        torch.cuda.synchronize()
        return [o.detach().cpu().numpy() for o in out] + [t[k].grad.cpu().numpy() for k in H.GRAD_KEYS]

    clean = run()
    monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
    poisoned = run()
    for a, b in zip(clean, poisoned):
        assert np.isfinite(b).all()
        np.testing.assert_array_equal(a, b)
