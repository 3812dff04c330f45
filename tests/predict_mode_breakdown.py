"""Mode prediction on one B200 (not collected by pytest): per shape (yeast, mirflickr and NUS-WIDE at S = 100 and 1000,
delicious, eurlex with Z = 3993 and Z = 10) and per input -- a planted model with about 5 labels per sample and the
worst case fx_out = 0 (E ~ 0.5 everywhere) --
  - call times of mpvae.predict, mpvae.score_sets with one set per row and mpvae.predict_mode: CUDA events, warm-up,
    median of 3 rounds with the callables alternated (a predict_mode call over 2 s is timed once instead);
  - the kernel times of one predict_mode call (torch.profiler, in a run of its own), split into the product (every
    kernel that is not a mode kernel), the row pass, the two scoring launches and the ascent;
  - the median ess and the median and largest number of flips.
python tests/predict_mode_breakdown.py --out DIR   -> DIR/r10_predict_mode.jsonl (one line for the card, one per shape)"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import synth                                                  # noqa: E402
from mpvae_b200.mpvae import predict, predict_mode, score_sets                 # noqa: E402
from tests.predict_breakdown import gpu_info                                  # noqa: E402
from tests.predict_ghk_breakdown import kernel_times, time_alternating        # noqa: E402
from tests.predict_sets_breakdown import planted_fx                           # noqa: E402
from tests.predict_sets_oracle import pack                                    # noqa: E402

SHAPES = [("yeast", 100, 128, 14, 14), ("yeast_s1000", 1000, 128, 14, 14), ("mirflickr", 100, 128, 38, 38),
          ("mirflickr_s1000", 1000, 128, 38, 38), ("nuswide", 100, 128, 81, 81), ("nuswide_s1000", 1000, 128, 81, 81),
          ("delicious", 100, 128, 983, 983), ("eurlex", 100, 1024, 3993, 3993), ("eurlex_z10", 100, 1024, 3993, 10)]
KERNELS = {"rows": "probit_mode_rows_kernel", "score": "mode_score_kernel", "ascent": "mode_ascent_kernel"}


def run_shape(name, S, B, L, Z, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    r = torch.from_numpy(inp["r_sqrt_sigma"]).to(dev)
    args = synth.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=7, noise_offset=3)
    out = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, **info, "inputs": {}}
    for kind, fx in (("planted_5_per_row", planted_fx(r, B, 5.0, seed=2).to(dev)),
                     ("worst_fx_zero", torch.zeros(B, L, device=dev))):
        with torch.no_grad():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            predict_mode(fx, r, args)
            e0.record()
            res = predict_mode(fx, r, args)
            e1.record()
            torch.cuda.synchronize()
            once = e0.elapsed_time(e1)
            bits = pack(res.sets[:, None])
            fns = {"predict": lambda: predict(fx, r, args), "score_sets_c1": lambda: score_sets(fx, r, bits, args)}
            if once < 2000.0:
                fns["predict_mode"] = lambda: predict_mode(fx, r, args)
            ms = time_alternating(fns)
            ms.setdefault("predict_mode", once)
            kt = kernel_times(lambda: predict_mode(fx, r, args))
        split = {k: sum(v for n, v in kt.items() if kn in n) for k, kn in KERNELS.items()}
        split["product"] = sum(v for n, v in kt.items() if not any(kn in n for kn in KERNELS.values()))
        fl = res.flips.double()
        out["inputs"][kind] = {
            "ms": ms, "kernel_ms": kt, "split_ms": split,
            "ess_median": float(res.ess.median()), "ess_min": float(res.ess.min()),
            "flips_median": float(fl.median()), "flips_max": int(fl.max()), "size_mean": float(res.size.double().mean()),
            "peak_allocated_gb": float(torch.cuda.max_memory_allocated(dev)) / 1e9}
        print(json.dumps({name: {kind: out["inputs"][kind]}}), flush=True)
        torch.cuda.reset_peak_memory_stats(dev)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_mode_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r10_predict_mode.jsonl")
    with open(path, "w") as f:
        f.write(json.dumps({"card": info, "torch": torch.__version__}) + "\n")
        for name, S, B, L, Z in SHAPES:
            if name not in a.shapes.split(","):
                continue
            rec = run_shape(name, S, B, L, Z, info)
            f.write(json.dumps(rec) + "\n")
            f.flush()


if __name__ == "__main__":
    main()
