"""Set prediction on one B200 (not collected by pytest): per shape (the five breakdown shapes of DESIGN §4, S = 100) and
per input -- a planted model with about 5 labels per sample (eurlex-like cardinality) and the worst case fx_out = 0
(E ~ 0.5, every label in some sample) --
  - call times of mpvae.predict, mpvae.sample_labels and mpvae.predict_sets with max_size unbounded and 64: CUDA
    events, warm-up, median of 3 rounds with the callables alternated;
  - the kernel times of the sample pass and of the decoder (torch.profiler, one call in a run of its own);
  - the sample pass's share of its bound: it reads nr and fx_out and writes S B L / 8 bytes of bits, over the HBM3e
    bandwidth of the HGX B200 data sheet (7.7 TB/s for one GPU);
  - the distribution of |U_b|, the labels set in any of a row's samples, which sets the decoder's work.
python tests/predict_sets_breakdown.py --out DIR   -> DIR/r09_predict_sets.jsonl (one line for the card, one per shape)"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpvae_b200 import synth                                                           # noqa: E402
from mpvae_b200.mpvae import predict, predict_sets, sample_labels, unpack_label_samples  # noqa: E402
from tests.predict_breakdown import gpu_info                                           # noqa: E402
from tests.predict_conditional_breakdown import SHAPES                                 # noqa: E402
from tests.predict_ghk_breakdown import kernel_times, time_alternating                 # noqa: E402

HBM_TBS = 7.7


def planted_fx(r, B, per_row, seed):
    """fx_out whose marginals put about `per_row` labels in a sample: Phi^-1(per_row / L) on the predictive scale."""
    L = r.shape[0]
    g = torch.Generator().manual_seed(seed)
    q = torch.full((L,), per_row / L, dtype=torch.float64)
    z = torch.special.ndtri(q) * torch.sqrt(1.0 + (r.double().cpu() ** 2).sum(1))
    return (z[None, :] + 0.3 * torch.randn(B, L, generator=g, dtype=torch.float64)).float()


def run_shape(name, S, B, L, Z, info):
    dev = torch.device("cuda", 0)
    inp = synth.loss_inputs(L, Z, B, S, seed=1, label_rate=max(0.05, 20.0 / L), with_noise=False)
    r = torch.from_numpy(inp["r_sqrt_sigma"]).to(dev)
    args = synth.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=7, noise_offset=3)
    out = {"shape": name, "S": S, "B": B, "L": L, "Z": Z, **info, "inputs": {}}
    ldn = (L + 3) // 4 * 4
    sample_bytes = S * B * ldn * 4 + B * L * 4 + B * S * ((L + 31) // 32) * 4
    for kind, fx in (("planted_5_per_row", planted_fx(r, B, 5.0, seed=2).to(dev)),
                     ("worst_fx_zero", torch.zeros(B, L, device=dev))):
        with torch.no_grad():
            bits = sample_labels(fx, r, args)
            nu = unpack_label_samples(bits, L).any(1).sum(1).double()
            card = unpack_label_samples(bits, L).sum(2).double()
            fns = {"predict": lambda: predict(fx, r, args),
                   "sample_labels": lambda: sample_labels(fx, r, args),
                   "predict_sets_max64": lambda: predict_sets(fx, r, args, max_size=64)}
            # the unbounded decoder on dense rows can take seconds: one call decides whether it joins the rounds
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            predict_sets(fx, r, args)
            e1.record()
            torch.cuda.synchronize()
            once = e0.elapsed_time(e1)
            if once < 2000.0:
                fns["predict_sets"] = lambda: predict_sets(fx, r, args)
            ms = time_alternating(fns)
            ms.setdefault("predict_sets", once)
            kt = kernel_times(lambda: predict_sets(fx, r, args)) if once < 2000.0 else {"single_call_ms": once}
            kt64 = kernel_times(lambda: predict_sets(fx, r, args, max_size=64))
        samp = sum(v for k, v in kt64.items() if "probit_sample_labels_kernel" in k)
        qs = torch.tensor([0.0, 0.5, 0.9, 1.0], dtype=torch.float64, device=nu.device)
        out["inputs"][kind] = {
            "ms": ms, "kernel_ms": kt, "kernel_ms_max64": kt64,
            "U_b": dict(zip(("min", "median", "p90", "max"), (float(v) for v in torch.quantile(nu, qs)))),
            "mean_labels_per_sample": float(card.mean()),
            "sample_pass": {"bytes": sample_bytes, "least_ms": sample_bytes / (HBM_TBS * 1e12) * 1e3, "ms": samp,
                            "share_of_bound": (sample_bytes / (HBM_TBS * 1e12) * 1e3) / samp if samp else None}}
        print(json.dumps({name: {kind: out["inputs"][kind]}}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_sets_breakdown measures on the GPU"
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "r09_predict_sets.jsonl")
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
