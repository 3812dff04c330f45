"""Conditional prediction against predict (not collected by pytest), one B200: per shape, mpvae.predict and
mpvae.predict_conditional on the same fx_out and noise keys, with 0 observed labels, 5 per row and 10 % of L per row.
  - call times: CUDA events, warm-up, median of 5 rounds with the callables alternated;
  - the row passes' time (the library's "row forward / finalize" profile slot) and the product's;
  - the median and minimum ESS per setting;
  - a bits check that the nothing-observed case equals predict.
python tests/predict_conditional_breakdown.py --out DIR   -> DIR/r05_predict_conditional.jsonl (one line per shape, one
for the card)"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import synth                                       # noqa: E402
from mpvae_b200.mpvae import predict, predict_conditional          # noqa: E402
from tests.predict_breakdown import gpu_info, kernel_ms, time_alternating   # noqa: E402

# (name, S, B, L, Z)
SHAPES = [("nuswide", 100, 128, 81, 81), ("mirflickr", 100, 128, 38, 38), ("delicious", 100, 128, 983, 983),
          ("eurlex", 100, 1024, 3993, 3993), ("eurlex_z10", 100, 1024, 3993, 10)]


def observed(B, L, k, y, seed):
    """int8 (B, L): k labels per row observed with their value in y, the rest -1."""
    g = torch.Generator().manual_seed(seed)
    idx = torch.argsort(torch.rand(B, L, generator=g), dim=1)[:, :k].to(y.device)
    obs = torch.full((B, L), -1, dtype=torch.int8, device=y.device)
    obs.scatter_(1, idx, y.to(torch.int8).gather(1, idx))
    return obs


def run_shape(name, S, B, L, Z, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in inp.items()}
    args = synth.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=7, noise_offset=3)
    settings = {"none": 0, "5_per_row": 5, "10pct": max(1, L // 10)}
    obs = {k: observed(B, L, n, t["y"], seed=n) for k, n in settings.items()}
    out = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, "observed_per_row": settings, **info}
    fns = {"predict": lambda: predict(t["fx_out"], t["r_sqrt_sigma"], args)}
    for k in settings:
        fns[f"conditional_{k}"] = (lambda o: lambda: predict_conditional(t["fx_out"], t["r_sqrt_sigma"], o, args))(obs[k])
    with torch.no_grad():
        res = {k: predict_conditional(t["fx_out"], t["r_sqrt_sigma"], o, args) for k, o in obs.items()}
        base = predict(t["fx_out"], t["r_sqrt_sigma"], args)
        out["none_bit_equal_to_predict"] = bool(torch.equal(res["none"].prob, base)
                                                and bool((res["none"].log_evidence == 0).all())
                                                and bool((res["none"].ess == S).all()))
        out["ess"] = {k: {"median": float(r.ess.median()), "min": float(r.ess.min())} for k, r in res.items()}
        out["ms"] = time_alternating(fns)
        out["ratio_to_predict"] = {k: v / out["ms"]["predict"] for k, v in out["ms"].items() if k != "predict"}
        out["kernel_ms"] = {k: kernel_ms(f) for k, f in fns.items()}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_conditional_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r05_predict_conditional.jsonl")
    with open(path, "w") as f:
        f.write(json.dumps({"card": info, "torch": torch.__version__}) + "\n")
        for name, S, B, L, Z in SHAPES:
            if name not in a.shapes.split(","):
                continue
            rec = run_shape(name, S, B, L, Z, info)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
