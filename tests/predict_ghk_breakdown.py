"""The GHK conditional prediction against the importance path (not collected by pytest), one B200: per shape (the five
BASELINE shapes, S = 100) and per observed share (0, 5 per row, 10 % and 50 % of L), mpvae.predict_conditional_ghk and
mpvae.predict_conditional on the same fx_out, R and noise keys.
  - call times: CUDA events, warm-up, median of 3 rounds with the two callables alternated;
  - each GHK kernel's time (torch.profiler, one call in a run of its own), its work from the observed counts and its
    share of the bound that governs it: fp64 FMA for the factor and the chain (37 TFLOP/s: the HGX B200 data sheet's
    FP64 figure for one GPU), fp32 CUDA-core FMA for the update (148 SMs x 128 lanes x 2 x the card's max SM clock);
  - median and minimum ESS of both estimators;
  - a bits check that the nothing-observed case equals predict.
python tests/predict_ghk_breakdown.py --out DIR   -> DIR/r07_predict_ghk.jsonl (one line for the card, one per shape)"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import synth                                                          # noqa: E402
from mpvae_b200.mpvae import label_gram, predict, predict_conditional, predict_conditional_ghk   # noqa: E402
from tests.predict_breakdown import gpu_info                                          # noqa: E402
from tests.predict_conditional_breakdown import SHAPES, observed                      # noqa: E402

FP64_TFLOPS = 37.0


def time_alternating(fns, reps=3):
    """Median ms per call, callables alternated round by round; n calls per window sized to ~0.2 s."""
    n = {}
    for k, f in fns.items():
        f()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        f()
        torch.cuda.synchronize()
        n[k] = max(1, min(10, int(0.2 / max(time.perf_counter() - t0, 1e-6))))
    rec = {k: [] for k in fns}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for k, f in fns.items():
            e0.record()
            for _ in range(n[k]):
                f()
            e1.record()
            torch.cuda.synchronize()
            rec[k].append(e0.elapsed_time(e1) / n[k])
    return {k: sorted(v)[len(v) // 2] for k, v in rec.items()}


def kernel_times(fn):
    """ms per kernel name of one call (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" or getattr(ev, "device_time_total", 0) > 0:
            name = ev.key.replace("(anonymous namespace)::", "").replace("mpv::", "").split("(")[0].split("<")[0]
            ms = getattr(ev, "device_time_total", 0.0) / 1e3
            if ms > 0:
                out[name] = out.get(name, 0.0) + ms
    return out


def work(obs, S, L):
    """fp64 MACs of the factor (n^3 / 6 per row) and the chain (1.5 S n^2: two forward dots and one backward dot per
    step), fp32 MACs of the update (S n L per row)."""
    n = ((obs == 0) | (obs == 1)).sum(1).double()
    return {"factor_fp64_mac": float((n ** 3 / 6).sum()), "chain_fp64_mac": float((1.5 * S * n ** 2).sum()),
            "update_fp32_mac": float((S * n * L).sum()), "max_observed": int(n.max()), "mean_observed": float(n.mean())}


def run_shape(name, S, B, L, Z, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in inp.items()}
    args = synth.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=7, noise_offset=3)
    settings = {"none": 0, "5_per_row": min(5, L), "10pct": max(1, L // 10), "50pct": max(1, L // 2)}
    fp32_tflops = 148 * 128 * 2 * info["sm_mhz"] * 1e6 / 1e12
    out = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, "observed_per_row": settings, **info,
           "bounds_tflops": {"fp64_fma": FP64_TFLOPS, "fp32_fma": fp32_tflops}, "settings": {}}
    with torch.no_grad():
        base = predict(t["fx_out"], t["r_sqrt_sigma"], args)
        for k, nobs in settings.items():
            o = observed(B, L, nobs, t["y"], seed=nobs)
            imp = lambda: predict_conditional(t["fx_out"], t["r_sqrt_sigma"], o, args)
            ghk = lambda: predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"], o, args)
            ri, rg = imp(), ghk()
            rec = {"ess": {"importance": {"median": float(ri.ess.median()), "min": float(ri.ess.min())},
                           "ghk": {"median": float(rg.ess.median()), "min": float(rg.ess.min())}},
                   "ghk_finite": bool(torch.isfinite(rg.prob).all() and torch.isfinite(rg.log_evidence).all())}
            if nobs == 0:
                rec["none_bit_equal_to_predict"] = bool(torch.equal(rg.prob, base) and bool((rg.log_evidence == 0).all())
                                                        and bool((rg.ess == S).all()))
            rec["ms"] = time_alternating({"importance": imp, "ghk": ghk})
            rec["ghk_over_importance"] = rec["ms"]["ghk"] / rec["ms"]["importance"]
            rec["ms_gram"] = time_alternating({"label_gram": lambda: label_gram(t["r_sqrt_sigma"], args)})["label_gram"]
            kt = kernel_times(ghk)
            rec["kernel_ms"] = kt
            w = work(o, S, L)
            rec["work"] = w
            share = {}
            for kern, key, peak in (("ghk_factor_kernel", "factor_fp64_mac", FP64_TFLOPS),
                                    ("ghk_chain_kernel", "chain_fp64_mac", FP64_TFLOPS),
                                    ("ghk_update_kernel", "update_fp32_mac", fp32_tflops)):
                ms = sum(v for n, v in kt.items() if kern in n)
                if ms > 0:
                    least = 2 * w[key] / (peak * 1e12) * 1e3
                    share[kern] = {"ms": ms, "least_ms": least, "share_of_bound": least / ms}
            rec["share"] = share
            out["settings"][k] = rec
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_ghk_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r07_predict_ghk.jsonl")
    with open(path, "w") as f:
        f.write(json.dumps({"card": info, "torch": torch.__version__}) + "\n")
        for name, S, B, L, Z in SHAPES:
            if name not in a.shapes.split(","):
                continue
            rec = run_shape(name, S, B, L, Z, info)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
            f.flush()


if __name__ == "__main__":
    main()
