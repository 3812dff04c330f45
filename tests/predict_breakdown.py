"""Label-free prediction against the test-mode loss forward (not collected by pytest), one B200:
  (a) compute_loss(mode='test') under no_grad vs mpvae.predict on the same fx_out and noise keys,
  (b) end to end from features: VAE.forward + compute_loss vs VAE.feat_forward + predict,
  (c) the library's per-slot kernel times (mpvae_profile) of both,
plus the predict row kernel's time against its two bounds and a bit-equality check of the two predictions.
python tests/predict_breakdown.py --out DIR   -> DIR/r03_predict_breakdown.jsonl (one line per shape, one for the card)"""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import _lib, synth                      # noqa: E402
from mpvae_b200.mpvae import VAE, compute_loss, predict  # noqa: E402

# (name, S, B, L, Z, feature_dim)
SHAPES = [("nuswide", 100, 128, 81, 81, 128), ("mirflickr", 100, 128, 38, 38, 1000), ("delicious", 100, 128, 983, 983, 500),
          ("eurlex", 100, 1024, 3993, 3993, 5000), ("eurlex_z10", 100, 1024, 3993, 10, 5000)]
HBM_BYTES_PER_S = 7.7e12           # B200 data sheet, one GPU
# SASS instructions per cell of probit_predict_rows_kernel<false>'s main loop (cuobjdump -sass: ~274 instructions per
# iteration of 2 samples x 4 labels, loads and loop control included), for the issue bound: 4 warp-instructions per SM
# and clock
INSTR_PER_CELL = 274 / 8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = (s.strip() for s in q.split(","))
    return {"gpu": name, "power_limit": power, "clocks_max_sm": clk, "sm_mhz": float(clk.split()[0])}


def time_alternating(fns, reps=5, n=10):
    """Median ms per call of each callable, the callables alternated round by round (shared host: compare in one run)."""
    for f in fns.values():
        for _ in range(2):
            f()
    torch.cuda.synchronize()
    rec = {k: [] for k in fns}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for k, f in fns.items():
            e0.record()
            for _ in range(n):
                f()
            e1.record()
            torch.cuda.synchronize()
            rec[k].append(e0.elapsed_time(e1) / n)
    return {k: float(np.median(v)) for k, v in rec.items()}


def kernel_ms(fn, n=5):
    fn()
    torch.cuda.synchronize()
    _lib.profile(True)
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    out = {k: ms / n for k, (ms, _) in _lib.profile_read().items()}
    _lib.profile(False)
    return out


def run_shape(name, S, B, L, Z, F, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in inp.items()}
    args = SimpleNamespace(feature_dim=F, label_dim=L, latent_dim=50, z_dim=Z, keep_prob=0.5, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=10, n_test_sample=S, mode="test", nll_coeff=0.5, c_coeff=10.0,
                           noise_seed=7, noise_offset=3)
    loss = lambda: compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                                t["r_sqrt_sigma"], args)
    pred = lambda: predict(t["fx_out"], t["r_sqrt_sigma"], args)
    out = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, "feature_dim": F, **info}
    with torch.no_grad():
        out["bit_equal"] = bool(torch.equal(loss()[6], pred()))
        out["a_ms"] = time_alternating({"loss_forward_test": loss, "predict": pred})
        np.random.seed(4)
        torch.manual_seed(0)
        model = VAE(args).to(dev).eval()
        x = torch.from_numpy(synth.features(B, F, np.random.RandomState(2))).to(dev)
        e2e_loss = lambda: compute_loss(t["y"], *model(t["y"], x), model.r_sqrt_sigma, args)
        e2e_pred = lambda: predict(model.feat_forward(x)[0], model.r_sqrt_sigma, args)
        out["b_ms"] = time_alternating({"forward_and_loss": e2e_loss, "feat_forward_and_predict": e2e_pred})
        out["c_kernel_ms"] = {"loss_forward_test": kernel_ms(loss), "predict": kernel_ms(pred)}
    # the predict row kernel (or the one-launch small-regime kernel) against its bounds
    kp = out["c_kernel_ms"]["predict"]
    row_key = next(k for k in kp if k.startswith("row forward") or k.startswith("fused small"))
    t_row = kp[row_key]
    ldn = (L + 3) & ~3
    hbm_ms = (S * B * ldn * 4 + 2 * B * L * 4) / HBM_BYTES_PER_S * 1e3
    issue_ms = S * B * L * INSTR_PER_CELL / 32 / (148 * 4 * info["sm_mhz"] * 1e6) * 1e3
    out["row_kernel"] = {"slot": row_key, "ms": t_row, "hbm_bound_ms": hbm_ms, "issue_bound_ms": issue_ms,
                         "bound": "HBM" if hbm_ms >= issue_ms else "issue", "share_of_bound": max(hbm_ms, issue_ms) / t_row,
                         "working_set_bytes": S * B * ldn * 4, "exceeds_L2": S * B * ldn * 4 > 126e6}
    if row_key.startswith("fused small"):
        out["row_kernel"]["note"] = "one launch per call incl. R staging, Philox and the FMA chain: not a streaming kernel"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r03_predict_breakdown.jsonl")
    with open(path, "w") as f:
        f.write(json.dumps({"card": info, "torch": torch.__version__}) + "\n")
        for name, S, B, L, Z, F in SHAPES:
            if name not in a.shapes.split(","):
                continue
            rec = run_shape(name, S, B, L, Z, F, info)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
