"""Masked loss against the unmasked loss (not collected by pytest), one B200: per BASELINE shape, one training loss step
(compute_loss forward + backward from total_loss, n_train_sample = 10, library Philox noise) in four settings: no mask,
an all-ones mask, 50 % and 10 % of the labels observed (random cells).
  - step times: CUDA events, warm-up, median of 7 rounds with the settings alternated;
  - the library's per-slot kernel times (row forward / finalize, row backward, fused small-regime kernels, products);
  - a bits check that the all-ones mask gives the unmasked outputs and gradients.
python tests/masked_loss_breakdown.py --out DIR   -> DIR/r06_masked_loss.jsonl (one line per shape, one for the card)"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import synth                                       # noqa: E402
from mpvae_b200.mpvae import compute_loss                          # noqa: E402
from tests.predict_breakdown import gpu_info, kernel_ms, time_alternating   # noqa: E402

# (name, S, B, L, Z): the training shapes of BASELINE.json
SHAPES = [("yeast", 10, 128, 14, 14), ("mirflickr", 10, 128, 38, 38), ("nuswide", 10, 128, 81, 81),
          ("delicious", 10, 128, 983, 983), ("eurlex", 10, 1024, 3993, 3993)]
LEAVES = ("fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma")


def run_shape(name, S, B, L, Z, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in inp.items()}
    leaves = {k: t[k].clone().requires_grad_(True) for k in LEAVES}
    args = synth.make_args(L, Z, n_train_sample=S, mode="train", noise_seed=7, noise_offset=3)
    g = torch.Generator().manual_seed(5)
    masks = {"unmasked": None, "all_ones": torch.ones(B, L, dtype=torch.bool, device=dev),
             "observed_50pct": (torch.rand(B, L, generator=g) < 0.5).to(dev),
             "observed_10pct": (torch.rand(B, L, generator=g) < 0.1).to(dev)}

    def step(mask):
        for v in leaves.values():
            v.grad = None
        kw = {} if mask is None else {"label_mask": mask}
        out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, **kw)
        out[0].backward()
        return out

    fns = {k: (lambda m: lambda: step(m))(m) for k, m in masks.items()}
    rec = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, "mask_bytes": B * L, **info}
    o0 = [o.detach().clone() for o in step(None)]
    g0 = {k: leaves[k].grad.clone() for k in LEAVES}
    o1 = [o.detach().clone() for o in step(masks["all_ones"])]
    g1 = {k: leaves[k].grad.clone() for k in LEAVES}
    rec["all_ones_bit_equal"] = all(torch.equal(a.nan_to_num(), b.nan_to_num()) for a, b in zip(o0, o1)) and \
        all(torch.equal(g0[k].nan_to_num(), g1[k].nan_to_num()) for k in LEAVES)
    rec["ms"] = time_alternating(fns, reps=7)
    rec["ratio_to_unmasked"] = {k: v / rec["ms"]["unmasked"] for k, v in rec["ms"].items() if k != "unmasked"}
    rec["kernel_ms"] = {k: kernel_ms(f) for k, f in fns.items()}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "masked_loss_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r06_masked_loss.jsonl")
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
