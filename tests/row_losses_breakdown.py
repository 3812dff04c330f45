"""Per-row losses against the batch means (not collected by pytest), one B200: per shape, one training loss step
(compute_loss forward + backward, n_train_sample = 10, library Philox noise) with reduction='mean' (cotangent 1 on
total_loss) and with reduction='none' (cotangent 1 / B on every row's total_loss, the same objective).
  - step times: CUDA events, warm-up, median of 7 rounds with the two settings alternated;
  - the library's per-slot kernel times (row forward / finalize, gxs bound, row backward, fused small-regime kernels,
    products);
  - a check that the mean over the rows of every per-row output is the batch output (largest relative difference).
python tests/row_losses_breakdown.py --out DIR   -> DIR/r16_row_losses.jsonl (one line for the card, one per shape)"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import synth                                       # noqa: E402
from mpvae_b200.mpvae import compute_loss                          # noqa: E402
from tests.predict_breakdown import gpu_info, kernel_ms, time_alternating   # noqa: E402

# (name, S, B, L, Z): a small training shape of BASELINE.json and the two dense ones
SHAPES = [("mirflickr", 10, 128, 38, 38), ("delicious", 10, 128, 983, 983), ("eurlex", 10, 1024, 3993, 3993)]
LEAVES = ("fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma")


def run_shape(name, S, B, L, Z, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in inp.items()}
    leaves = {k: t[k].clone().requires_grad_(True) for k in LEAVES}
    args = synth.make_args(L, Z, n_train_sample=S, mode="train", noise_seed=7, noise_offset=3)
    per_row = torch.full((B,), 1.0 / B, device=dev)

    def step(reduction):
        for v in leaves.values():
            v.grad = None
        out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, reduction=reduction)
        out[0].backward(per_row if reduction == "none" else None)
        return out

    fns = {r: (lambda r: lambda: step(r))(r) for r in ("mean", "none")}
    rec = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, **info}
    om = [o.detach().clone() for o in step("mean")]
    on = [o.detach().clone() for o in step("none")]
    rec["max_rel_diff_row_mean_vs_mean"] = max(
        abs(float(on[i].double().mean()) - float(om[i])) / max(1.0, abs(float(om[i]))) for i in range(6))
    rec["predictions_bit_equal"] = torch.equal(om[6], on[6]) and torch.equal(om[7], on[7])
    rec["ms"] = time_alternating(fns, reps=7)
    rec["ratio_none_to_mean"] = rec["ms"]["none"] / rec["ms"]["mean"]
    rec["kernel_ms"] = {k: kernel_ms(f) for k, f in fns.items()}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "row_losses_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r16_row_losses.jsonl")
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
