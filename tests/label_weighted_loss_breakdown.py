"""Label-weighted loss against the unweighted loss (not collected by pytest), one B200: per BASELINE shape, one training
loss step (compute_loss forward + backward from total_loss, n_train_sample = 10, library Philox noise) without weights,
with all-ones label weights, with random label weights (10 % of them 0), and with random label weights combined with a
label mask (70 % observed) and random row weights.
  - step times: CUDA events, warm-up, median of 7 rounds with the settings alternated;
  - the library's per-slot kernel times (row forward / finalize, gxs bound, row backward, fused small-regime kernels,
    products);
  - a bits check that all-ones label weights give the unweighted outputs and gradients.
python tests/label_weighted_loss_breakdown.py --out DIR   -> DIR/r14_label_weighted_loss.jsonl (one line for the card,
one per shape)"""
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
    pos, neg = torch.rand(L, generator=g) * 4.0, torch.rand(L, generator=g) * 2.0
    pos[torch.rand(L, generator=g) < 0.1] = 0.0
    neg[torch.rand(L, generator=g) < 0.1] = 0.0
    pos, neg = pos.to(dev), neg.to(dev)
    mask = (torch.rand(B, L, generator=g) < 0.7).to(dev)
    rows = (torch.rand(B, generator=g) * 2.0).to(dev)
    ones = torch.ones(L, device=dev)
    weights = {"unweighted": {}, "all_ones": {"pos_weight": ones, "neg_weight": ones},
               "random": {"pos_weight": pos, "neg_weight": neg},
               "masked_row_weighted": {"label_mask": mask, "row_weight": rows},
               "random_masked_row_weighted": {"pos_weight": pos, "neg_weight": neg, "label_mask": mask, "row_weight": rows}}

    def step(kw):
        for v in leaves.values():
            v.grad = None
        out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, **kw)
        out[0].backward()
        return out

    fns = {k: (lambda w: lambda: step(w))(w) for k, w in weights.items()}
    rec = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, **info}
    o0 = [o.detach().clone() for o in step({})]
    g0 = {k: leaves[k].grad.clone() for k in LEAVES}
    o1 = [o.detach().clone() for o in step(weights["all_ones"])]
    g1 = {k: leaves[k].grad.clone() for k in LEAVES}
    rec["all_ones_bit_equal"] = all(torch.equal(a.nan_to_num(), b.nan_to_num()) for a, b in zip(o0, o1)) and \
        all(torch.equal(g0[k].nan_to_num(), g1[k].nan_to_num()) for k in LEAVES)
    rec["ms"] = time_alternating(fns, reps=7)
    rec["ratio_to_unweighted"] = {k: v / rec["ms"]["unweighted"] for k, v in rec["ms"].items() if k != "unweighted"}
    rec["kernel_ms"] = {k: kernel_ms(f) for k, f in fns.items()}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "label_weighted_loss_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r14_label_weighted_loss.jsonl")
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
