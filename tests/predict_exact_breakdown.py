"""Closed-form prediction against the Monte-Carlo predict (not collected by pytest), one B200:
  (a) per call: mpvae.predict at S = 100 and S = 10 000 (eurlex at B = 128, where its nr fits), the scale preparation
      (predictive_scale) and mpvae.predict_exact (scale pass included), alternated round by round;
  (b) the pairs kernel on every NUS-WIDE pair x B = 1024 and on 1 M random eurlex pairs x B = 128, plus the rho
      preparation, in cells/s against a fp64 issue bound derived from the kernel's SASS;
  (c) accuracy on a synthetic trained model: the share of cells on the other side of 0.5 and the p@1 disagreement of
      S = 100 predict against predict_exact.
python tests/predict_exact_breakdown.py --out DIR   -> DIR/r04_predict_exact.jsonl (one line for the card, one per record)"""
import argparse
import json
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import mpvae, probit, synth            # noqa: E402
from tests.predict_breakdown import gpu_info, time_alternating   # noqa: E402

# (name, B, L, Z): the shapes of predict_breakdown.py; eurlex's S = 10 000 leg runs at B = 128
SHAPES = [("nuswide", 128, 81, 81), ("mirflickr", 128, 38, 38), ("delicious", 128, 983, 983), ("eurlex", 1024, 3993, 3993),
          ("eurlex_b128", 128, 3993, 3993)]
# fp64 issue bound of predict_pairs_kernel, DERIVED (not measured): cuobjdump -sass of predict_pairs_kernel<false>
# (sm_100a) holds 4029 fp64-pipe instructions (DFMA 2973, DMUL 534, DADD 386, DSETP 136) over 58 unrolled node bodies
# (the 6-, 12- and 20-node rules of |rho| < 0.925 and the 20 nodes of the tail branch): ~69 per node.  A cell of a pair
# with n nodes issues ~69 n of them; the SM's fp64 pipe takes 64 per clock (HGX B200 data sheet: 296 TFLOP/s FP64 for
# eight GPUs = 37 per GPU, i.e. 64 FMA per SM and clock at 1.965 GHz on 148 SMs).
FP64_PER_NODE = 4029 / 58
FP64_PER_SM_CLK = 64


def _args(L, Z, S):
    return SimpleNamespace(label_dim=L, z_dim=Z, n_test_sample=S, mode="test", noise_seed=7, noise_offset=3, mpvae_flags=0)


def nodes_per_pair(rho):
    a = rho.abs()
    return torch.where(a < 0.3, 6, torch.where(a < 0.75, 12, 20)).double()


def timing(name, B, L, Z):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, 1, seed=1, with_noise=False)
    fx, r = torch.from_numpy(inp["fx_out"]).to(dev), torch.from_numpy(inp["r_sqrt_sigma"]).to(dev)
    r32 = r.float()
    fns = {"predict_exact": lambda: mpvae.predict_exact(fx, r, _args(L, Z, 100)),
           "scale": lambda: probit.predictive_scale(r32)}
    fns["predict_S100"] = lambda: mpvae.predict(fx, r, _args(L, Z, 100))
    if name != "eurlex":
        fns["predict_S10000"] = lambda: mpvae.predict(fx, r, _args(L, Z, 10_000))
    with torch.no_grad():
        ms = time_alternating(fns, reps=5, n=10 if "predict_S10000" not in fns else 3)
    out = {"shape": name, "B": B, "L": L, "Z": Z, "ms": ms}
    if "predict_S100" in ms:
        out["predict_exact_speedup_vs_S100"] = ms["predict_S100"] / ms["predict_exact"]
    if "predict_S10000" in ms:
        out["predict_exact_speedup_vs_S10000"] = ms["predict_S10000"] / ms["predict_exact"]
    out["exact_bytes"] = 2 * B * L * 4 + L * Z * 4 + L * 8
    out["exact_hbm_bound_ms"] = out["exact_bytes"] / 7.7e12 * 1e3
    return out


def pairs_timing(name, B, L, Z, pairs, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, 1, seed=2, with_noise=False)
    fx, r = torch.from_numpy(inp["fx_out"]).to(dev), torch.from_numpy(inp["r_sqrt_sigma"]).to(dev)
    args = _args(L, Z, 100)
    with torch.no_grad():
        pp = mpvae.PairPredictor(r, pairs, args)
        ms = time_alternating({"pairs": lambda: pp(fx), "prepare": lambda: mpvae.PairPredictor(r, pairs, args)},
                              reps=5, n=3)
        nodes = nodes_per_pair(pp.rho).sum().item() * B
    cells = B * pp.pairs.shape[0]
    bound_ms = nodes * FP64_PER_NODE / (FP64_PER_SM_CLK * 148 * info["sm_mhz"] * 1e6) * 1e3
    return {"pairs": name, "B": B, "L": L, "Z": Z, "P": pp.pairs.shape[0], "ms": ms, "cells_per_s": cells / ms["pairs"] * 1e3,
            "fp64_issue_bound_ms_derived": bound_ms, "share_of_derived_bound": bound_ms / ms["pairs"],
            "rho_abs_max": pp.rho.abs().max().item(), "mean_nodes_per_cell": nodes / cells}


def accuracy():
    """A yeast-sized synthetic model trained a few epochs: S = 100 predict vs predict_exact on held-out rows."""
    from mpvae_b200.infer import predict_proba
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    from tests.test_predict_gpu import _yeast_args, _yeast_data
    dev = torch.device("cuda", 0)
    args = _yeast_args()
    x, y = _yeast_data(1500)
    np.random.seed(4)
    torch.manual_seed(0)
    vae = mpvae.VAE(args).to(dev)
    opt = torch.optim.Adam(vae.parameters(), lr=1e-3, weight_decay=1e-5)
    step = DataParallelStep(vae, opt, torch.optim.lr_scheduler.StepLR(opt, 45, 0.5), args, clip_norm=100.0)
    for _ in range(12):
        train_one_epoch(step, x[:1050], y[:1050], 128, torch.randperm(1050, device=dev))
    vae._reparameterize = lambda mu, logvar: mu         # the same fx_out for both
    xv = x[1050:]
    exact, _ = predict_proba(vae, xv, None, args, predict_fn=mpvae.predict_exact)
    mc, _ = predict_proba(vae, xv, None, args)          # args.n_test_sample = 100
    mc4, _ = predict_proba(vae, xv, None, SimpleNamespace(**{**vars(args), "n_test_sample": 10_000}))
    flip = lambda a: float(((a >= 0.5) != (exact >= 0.5)).float().mean())
    p1 = lambda a: float((a.argmax(1) != exact.argmax(1)).float().mean())
    return {"accuracy": "yeast-sized synthetic model, 12 epochs, 450 held-out rows x 14 labels",
            "cells_across_0.5_S100": flip(mc), "p_at_1_disagreement_S100": p1(mc),
            "cells_across_0.5_S10000": flip(mc4), "p_at_1_disagreement_S10000": p1(mc4),
            "max_abs_diff_S100": float((mc - exact).abs().max()), "max_abs_diff_S10000": float((mc4 - exact).abs().max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_exact_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r04_predict_exact.jsonl")
    g = torch.Generator().manual_seed(0)
    with open(path, "w") as f:
        def emit(rec):
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
        emit({"card": info, "torch": torch.__version__})
        for shape in SHAPES:
            emit(timing(*shape))
        emit(pairs_timing("nuswide_all", 1024, 81, 81, mpvae.all_pairs(81), info))
        emit(pairs_timing("eurlex_1M_random", 128, 3993, 3993, torch.randint(0, 3993, (1 << 20, 2), generator=g), info))
        emit(accuracy())


if __name__ == "__main__":
    main()
