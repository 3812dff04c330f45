"""Measurement helper (not a test): per-kernel device times of the loss step from the library's own CUDA-event records
(mpvae_profile*), with the noise drawn by the product kernel's math warps and by a kernel of its own.

    python tests/step_breakdown.py [--workload eurlex] [--z Z] [--batch B] [--steps 20] [--external-noise]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mpvae_b200 import _lib, synth
from mpvae_b200 import mpvae as M


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="eurlex")
    ap.add_argument("--z", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--external-noise", action="store_true")
    a = ap.parse_args()
    sh = synth.SHAPES[a.workload]
    L, Z, B, S = sh.label_dim, a.z or sh.z_dim, a.batch or sh.batch, sh.n_sample
    dev = torch.device("cuda:0")
    inp = synth.loss_inputs(L, Z, B, S, seed=100, label_rate=sh.label_rate, with_noise=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in inp.items()}
    r32 = t.pop("r_sqrt_sigma").float().requires_grad_(True)
    noise = torch.randn(S, B, Z, device=dev) if a.external_noise else None
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    for name, flags in (("default", 0), ("separate_noise_kernel", _lib.FLAG_SEPARATE_NOISE)):
        args = synth.make_args(L, Z, n_train_sample=S, n_test_sample=S, mode=sh.mode, mpvae_flags=flags, noise_seed=1)

        def step(i):
            args.noise_offset = i
            leaves = {k: (v if k == "y" else v.detach().requires_grad_(True)) for k, v in t.items()}
            r32.grad = None
            out = M.compute_loss(leaves["y"], leaves["fe_out"], leaves["fe_mu"], leaves["fe_logvar"], leaves["fx_out"],
                                 leaves["fx_mu"], leaves["fx_logvar"], r32, args, **({"noise": noise} if noise is not None else {}))
            if sh.mode == "train":
                out[0].backward()
            return out

        for i in range(5):
            step(i)
        torch.cuda.synchronize()
        evs = []
        for i in range(a.steps):
            flush.add_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); step(10 + i); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in evs)
        _lib.profile(True)
        for i in range(a.steps):
            flush.add_(1.0)
            out = step(100 + i)
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile(False)
        print(json.dumps({"variant": name, "workload": f"{a.workload} S{S} B{B} L{L} Z{Z}" + (" external noise" if noise is not None else ""),
                          "step_ms_median": ms[len(ms) // 2], "step_ms_min": ms[0], "loss": float(out[0]),
                          "kernel_ms": {k: round(v[0] / v[1], 4) for k, v in prof.items()}}), flush=True)


if __name__ == "__main__":
    main()
