#!/usr/bin/env python
"""bench.py -- probit-ELBO fwd+bwd throughput (label-samples/s) on B200, BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload eurlex] [--z Z] [--scaling weak|strong]
                    [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: draw the (S,B,Z) noise (Philox, on device), the forward of
compute_loss (mpvae.py:145-210) and its full backward to logits / R / mu / logvar; at N > 1 the step ends with the sum
of g_R over the ranks (the path's one exchange).  `--scaling weak` (default): every rank owns the workload's B rows;
`--scaling strong`: the workload's B rows are the GLOBAL batch, rank r owns rows [r B/N, (r+1) B/N) (BASELINE.json
configs[4], SURVEY 8e); a run at N > 1 also reports the other mode as a short leg (`strong_scaling` / `weak_scaling`).
`value` times the step with the inputs resident in HBM; `e2e` times the same call through the public
`mpvae_b200.compute_loss` API starting from pinned HOST buffers (H2D of the step's inputs, D2H of the loss and of the
step's eight metrics inside the timed region).  Prints ONE JSON line (rank 0).

`--dump-outputs DIR` writes what the last step timed for `value` returned: compute_loss's eight outputs and, for a
training workload, the gradients of the loss with respect to its seven differentiable inputs (`grad_<input>`), as
DIR/<name>.npy.  Inputs and noise are seeded, so runs with the same arguments see the same inputs and two builds can be
compared output for output.

`--impl reference` times the reference's own CPU implementation instead: the UNMODIFIED compute_loss of
/root/reference/mpvae.py, placed under oracle/_ref/ by oracle/make_ref.py (the oracle port when that copy is absent),
on all host cores, on a bounded row sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "probit-ELBO fwd+bwd label-samples/s"
UNIT = "label-samples/s"
L2_BYTES = 126 * 1024 * 1024
ROW_KEYS = ["y", "fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar"]
# compute_loss's 8-tuple, in order
OUT_NAMES = ["total_loss", "nll_loss", "nll_loss_x", "c_loss", "c_loss_x", "kl_loss", "indiv_prob", "indiv_prob_label"]
# per dumped array: 8 outputs + 7 gradients of at most 4 MB each keep a dump under 64 MB
DUMP_MAX_BYTES = 4 << 20

# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
# captures under profiles/ ((L, Z, S*B rows, fused row forward) -> bytes)
TRAFFIC = {
    # profiles/r02_final_ncu_full_summary.txt: 428.47 MB read + 226.55 MB written by the nt product that also draws its
    # noise plane (round 1, separate Philox kernel: 769.18 MB, profiles/r01_final_ncu_full_summary.txt)
    (3993, 3993, 10240, False): 655.02e6,
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="eurlex", help="one of mpvae_b200.synth.SHAPES")
    ap.add_argument("--z", type=int, default=None, help="rank of R (default: the workload's, z_dim = label_dim)")
    ap.add_argument("--batch", type=int, default=None, help="rows of the workload's batch (default: the workload's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch rows per GPU; strong: --batch rows in total, sharded over the GPUs")
    ap.add_argument("--cpu-rows", type=int, default=None, help="rows of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true", help="skip the reference-on-this-GPU (torch CUDA ops) leg")
    ap.add_argument("--no-train-step", action="store_true", help="skip the full-training-step (steps/s) leg")
    ap.add_argument("--profile-host", action="store_true",
                    help="diagnostic: cProfile of 20 end-to-end steps on the host (top entries to stderr) after the timed legs")
    ap.add_argument("--engine", default="auto", choices=["auto", "fma", "tensor"])
    ap.add_argument("--fused-row-forward", action="store_true",
                    help="dense regime: run the row forward on math warps inside the product kernel (A/B; measured slower)")
    ap.add_argument("--serial-exchange", action="store_true",
                    help="N>1, peer exchange: sum g_R only after the g_R product instead of slab by slab beside it (A/B)")
    ap.add_argument("--fused-exchange", action="store_true",
                    help="N>1, peer exchange: sum g_R tile by tile inside the g_R product kernel instead of with the "
                         "stand-alone reduce kernel after it (A/B)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nvls", "nccl"],
                    help="N>1: how g_R is summed over ranks (peer = inside the backward over NVLink peer memory, "
                         "mpvae_b200.peer.PeerRing, falling back to nccl if the ring cannot be set up on every rank; "
                         "nccl = all-reduce after the backward)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (loss terms, probabilities, gradients; rank 0's) as "
                         "DIR/<name>.npy, arrays above %d MB as a fixed seeded sample" % (DUMP_MAX_BYTES >> 20))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        d["_source"] = "measured"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0,
            "_source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []          # (arrival time, csv line); only those inside [t0, t1] are reported
        self.proc = None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.monotonic()

    def mark_end(self):
        self.t1 = time.monotonic()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = self.t0 if self.t0 is not None else float("-inf")
        t1 = self.t1 if self.t1 is not None else float("inf")
        for when, ln in self.lines:
            if not (t0 <= when <= t1):
                continue          # nvidia-smi was started before the warm-up so that it is already looping here
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_outputs(tensors):
    """{name: device tensor} -> {name: float32/float64 numpy array}.  An array of more than DUMP_MAX_BYTES becomes a
    sample of its flattened elements, as many as fit in DUMP_MAX_BYTES, taken at positions drawn from a fixed seed: the
    same positions for the same shape and dtype, so two builds' dumps compare element for element."""
    import numpy as np
    import torch
    host, positions = {}, {}
    for name, t in tensors.items():
        t = t.detach()
        if t.dtype not in (torch.float32, torch.float64):
            t = t.float()
        n, cap = t.numel(), DUMP_MAX_BYTES // t.element_size()
        if n > cap:
            if (n, cap) not in positions:
                positions[n, cap] = torch.from_numpy(np.sort(np.random.RandomState(0).choice(n, cap, replace=False)))
            t = t.reshape(-1)[positions[n, cap].to(t.device)]
        host[name] = t.cpu().numpy()
    return host


def workload(a):
    from mpvae_b200 import synth
    sh = synth.SHAPES[a.workload]
    Z = a.z if a.z is not None else sh.z_dim
    B = a.batch if a.batch is not None else sh.batch
    return sh, sh.label_dim, Z, B, sh.n_sample


# ------------------------------------------------------------------------------------------ cost model (SURVEY 8d)
FP32_LANES = 148 * 128 * 2          # FMA lanes x 2 flop
XU_LANES = 148 * 16


def cost_model(S, B, L, Z, D, train, dense, passes, peaks):
    """T_min of one step from the ALGORITHMIC work of SURVEY.md 8(d), cost model v0: per label-sample 4Z + 200 fp32 flop
    and 10 special-function evaluations for fwd+bwd (2Z + 120 and 6 forward only); HBM 4(7BL + 8BD + 2LZ) bytes
    (4(5BL + 4BD + LZ) forward only).  Dense regime (Z, L >= 128): all flops against the split-precision tensor peak
    (bf16 burst / MMA passes per fp32-equivalent product), as the round-1 review recomputed it; otherwise the CUDA-core
    FP32 issue rate, the XU rate and HBM, whichever is slowest."""
    cells = float(S) * B * L
    flops = cells * ((4 * Z + 200) if train else (2 * Z + 120))
    xu = cells * (10 if train else 6)
    hbm = 4.0 * ((7 * B * L + 8 * B * D + 2 * L * Z) if train else (5 * B * L + 4 * B * D + L * Z))
    f_max = peaks["sm_max_mhz"] * 1e6
    t_fp32 = flops / (FP32_LANES * f_max)
    t_xu = xu / (XU_LANES * f_max)
    t_hbm = hbm / (peaks["hbm_gbs"] * 1e9)
    out = {"flops": flops, "xu_ops": xu, "hbm_bytes": hbm, "t_fp32_ms": t_fp32 * 1e3, "t_xu_ms": t_xu * 1e3, "t_hbm_ms": t_hbm * 1e3}
    if dense:
        t_tensor = flops / (peaks["bf16_tflops"] * 1e12 / passes)
        out["t_tensor_ms"] = t_tensor * 1e3
        out["t_min_ms"] = max(t_tensor, t_xu, t_hbm) * 1e3
        out["governs"] = "tensor"
    else:
        out["t_min_ms"] = max(t_fp32, t_xu, t_hbm) * 1e3
        out["governs"] = max((("fp32", t_fp32), ("xu", t_xu), ("hbm", t_hbm)), key=lambda kv: kv[1])[0]
    return out


# ------------------------------------------------------------------------------------------ CPU arm
def _reference_module():
    """The unmodified reference mpvae.py (oracle/_ref/, placed by oracle/make_ref.py) or None."""
    from oracle import make_ref
    if not os.path.exists(os.path.join(make_ref.OUT, "mpvae.py")):
        make_ref.make(quiet=True)          # build container only; on the GPU box the copy travels with the snapshot
    return make_ref.load()


def cpu_reference_step(L, Z, S, rows, seed=0, device="cpu", ref=None, train=True):
    """One fwd(+bwd) of the reference's algorithm on `rows` rows of the workload: the UNMODIFIED compute_loss when
    oracle/_ref/ is there (it draws its own torch.normal noise, mpvae.py:162), else the oracle port.  Returns seconds."""
    import torch
    from mpvae_b200 import synth
    inp = synth.loss_inputs(L, Z, rows, S, seed=seed + 1, label_rate=min(0.1, 20.0 / L), with_noise=ref is None)
    t = {k: torch.from_numpy(v).to(device) for k, v in inp.items()}
    sync = (lambda: torch.cuda.synchronize()) if str(device).startswith("cuda") else (lambda: None)
    if ref is not None:
        args = synth.make_args(L, Z, n_train_sample=S, n_test_sample=S, mode="train" if train else "test")
        leaves = [t[k].requires_grad_(train) for k in ("fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma")]
        sync()
        t0 = time.perf_counter()
        with torch.enable_grad() if train else torch.no_grad():
            out = ref.compute_loss(t["y"], leaves[0], leaves[1], leaves[2], leaves[3], leaves[4], leaves[5], leaves[6], args)
            if train:
                out[0].backward()
        sync()
        return time.perf_counter() - t0
    from oracle import probit_elbo_oracle as orc
    noise = t.pop("noise")
    sync()
    t0 = time.perf_counter()
    if train:
        orc.probit_elbo_with_grads(t, noise, 0.5, 10.0)
    else:
        with torch.no_grad():
            orc.probit_elbo(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                            t["r_sqrt_sigma"], noise, 0.5, 10.0)
    sync()
    return time.perf_counter() - t0


def torch_factorised_step(L, Z, S, rows, seed, device, train):
    """The reference's torch ops on `device` with the ranking loss in its exactly factorised form (oracle port)."""
    import torch
    from mpvae_b200 import synth
    from oracle import probit_elbo_oracle as orc
    inp = synth.loss_inputs(L, Z, rows, S, seed=seed + 1, label_rate=min(0.1, 20.0 / L), with_noise=False)
    t = {k: torch.from_numpy(v).to(device) for k, v in inp.items()}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    noise = torch.normal(0, 1, size=(S, rows, Z)).to(device)       # mpvae.py:162: drawn on the host, then copied
    if train:
        orc.probit_elbo_with_grads(t, noise, 0.5, 10.0, ranking="factorised")
    else:
        with torch.no_grad():
            orc.probit_elbo(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                            t["r_sqrt_sigma"], noise, 0.5, 10.0, ranking="factorised")
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def cpu_rows_for(L, Z, S, B, want=None):
    if want:
        return want
    # pairwise ranking loss materialises ~6 (S,rows,L,L) fp32 tensors (fwd+bwd): keep under ~24 GB and ~10-30 s
    per_row = 6 * S * L * L * 4
    return max(1, min(B, 128, int(24e9 // per_row)))


def cpu_kind(ref):
    return ("reference", "unmodified compute_loss of /root/reference/mpvae.py (oracle/_ref/)") if ref is not None \
        else ("port", "oracle port of mpvae.py:145-210")


def run_reference(a):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sh, L, Z, B, S = workload(a)
    train = sh.mode == "train"
    torch.set_num_threads(os.cpu_count())
    ref = _reference_module()
    kind, what = cpu_kind(ref)
    rows = cpu_rows_for(L, Z, S, B, a.cpu_rows)
    steps = max(1, a.steps)
    # bound the whole run to a few minutes: probe one step, then cap the step count
    t_probe = cpu_reference_step(L, Z, S, rows, ref=ref, train=train)
    budget = 150.0
    steps = max(1, min(steps, int(budget // max(t_probe, 1e-3))))
    warm = max(0, min(a.warmup, 1 if t_probe > 5 else 3))
    for i in range(warm):
        cpu_reference_step(L, Z, S, rows, seed=i, ref=ref, train=train)
    ts = [cpu_reference_step(L, Z, S, rows, seed=10 + i, ref=ref, train=train) for i in range(steps)]
    t = sum(ts) / len(ts)
    value = S * rows * L / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{sh.name}-shaped S{S} B{B} L{L} Z{Z} " + ("fwd+bwd" if train else "inference (forward, no_grad)"),
                   "S": S, "B_per_gpu": B, "L": L, "Z": Z, "note": "CPU arm runs a bounded row sample of this workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                         "sample": f"{rows} of {B} rows per step (the reference's O(L^2) ranking loss needs "
                                   f"{6 * S * L * L * 4 / 1e9:.1f} GB per row), {what} on torch CPU"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from mpvae_b200 import _lib, synth
    from mpvae_b200 import mpvae as M
    from mpvae_b200.metrics import batch_metrics_tensor
    from mpvae_b200.train import pack_labels, shard_rows, unpack_labels

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MPVAE_PEER_TIMEOUT_S", "30")     # a rank that never arrives ends the bench, it does not hang it
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sh, L, Z, B, S = workload(a)
    D = sh.latent_dim
    flags = {"auto": 0, "fma": _lib.FLAG_CONTRACT_FMA, "tensor": _lib.FLAG_CONTRACT_TENSOR}[a.engine]
    if a.fused_row_forward:
        flags |= _lib.FLAG_FUSED_FORWARD
    if a.fused_exchange:
        flags |= _lib.FLAG_FUSED_EXCHANGE
    if a.serial_exchange:
        flags |= _lib.FLAG_SERIAL_EXCHANGE
    infer = sh.mode == "test"       # BASELINE configs[2] (nuswide) is the test-time path: forward only, no_grad, S = n_test_sample
    dense = (Z >= 128 and L >= 128 and a.engine != "fma") or a.engine == "tensor"
    fused = dense and a.fused_row_forward and S <= 256
    passes = 2                      # library noise sits on the fp16 grid: one operand piece, two MMA passes
    peaks = measured_peaks()

    r_sqrt_sigma = torch.from_numpy(synth.loss_inputs(L, Z, 1, 1, seed=100, with_noise=False)["r_sqrt_sigma"]).to(dev)
    r32 = r_sqrt_sigma.float().requires_grad_(True)      # fp32 working copy of the (replicated) parameter
    flush = torch.empty(2 * L2_BYTES // 4, dtype=torch.float32, device=dev)
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    metrics_host = torch.empty(8, dtype=torch.float64).pin_memory()
    step_no = [0]

    class Leg:
        """One sharding of the workload: this rank's rows as pinned host and as device tensors + the args namespace."""

        def __init__(self, rows_global, lo, hi, seed):
            self.Bg, self.lo, self.hi = rows_global, lo, hi
            inp = synth.loss_inputs(L, Z, max(hi - lo, 1), S, seed=seed, label_rate=sh.label_rate, with_noise=False)
            self.host = {k: torch.from_numpy(inp[k][:hi - lo]).pin_memory() for k in ROW_KEYS}
            self.dev = {k: self.host[k].to(dev) for k in ROW_KEYS}
            # the {0,1} label matrix crosses PCIe as bits (1/32 of the fp32 size; packed once, the labels of a data set do
            # not change); mpvae_b200.train.unpack_labels restores the fp32 matrix on the device
            self.host["y"] = pack_labels(inp["y"][:hi - lo]).pin_memory()
            self.args = synth.make_args(L, Z, n_train_sample=S, n_test_sample=S, mode=sh.mode, nll_coeff=0.5, c_coeff=10.0,
                                        mpvae_flags=flags, noise_seed=1234, dp_global_batch=rows_global, dp_row0=lo)

    if a.scaling == "weak":
        main = Leg(B * world, rank * B, (rank + 1) * B, 100 + rank)
    else:
        lo, hi = shard_rows(B, rank, world)
        main = Leg(B, lo, hi, 100 + rank)
    if main.hi - main.lo < 1:
        raise RuntimeError(f"--scaling strong: batch {B} has no row for rank {rank} of {world}")

    # the path's one exchange: g_R summed over ranks.  Default: inside the backward over NVLink peer memory
    # (mpvae_b200.peer.PeerRing); --exchange nccl = an NCCL all-reduce after the backward.  If any rank fails to set
    # the ring up (CUDA IPC unavailable), every rank falls back to NCCL.
    ring = None
    if world > 1 and not infer and a.exchange in ("peer", "nvls"):
        from mpvae_b200.peer import NvlsRing, PeerRing
        try:
            # nvls: the chunk owners reduce inside the NVSwitch (multimem.ld_reduce / multimem.st)
            ring = (NvlsRing if a.exchange == "nvls" else PeerRing)(L, Z, dev)
        except Exception as e:          # noqa: BLE001 -- any failure means "use NCCL", decided collectively below
            print(f"[bench] rank {rank}: peer ring unavailable ({e}); NCCL exchange", file=sys.stderr)
            ring = None
        ok = torch.tensor([1 if ring is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0 and ring is not None:
            ring = None                 # (its buffers stay allocated; the process is short-lived)

    def one_step(leg, src, from_host, use_ring=True, noise=None, keep=None):
        """One step; `keep` (a dict), if given, receives what the step returns to its caller, by name."""
        args = leg.args
        args.noise_offset = step_no[0]
        args.peer_ring = ring if use_ring else None
        step_no[0] += 1
        t = src
        if t["y"].dtype != torch.float32:
            t = dict(t, y=unpack_labels(t["y"], L))   # the bit-packed labels of the host path: one unpack serves the loss and the metrics
        kw = {} if noise is None else {"noise": noise}
        if infer:
            with torch.no_grad():
                out = M.compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"],
                                     t["fx_logvar"], r32, args, **kw)
        else:
            leaves = {k: (t[k] if k == "y" else t[k].requires_grad_(True)) for k in ROW_KEYS}
            r32.grad = None
            out = M.compute_loss(leaves["y"], leaves["fe_out"], leaves["fe_mu"], leaves["fe_logvar"], leaves["fx_out"],
                                 leaves["fx_mu"], leaves["fx_logvar"], r32, args, **kw)
            out[0].backward()
            if world > 1:
                if ring is None or not use_ring:
                    dist.all_reduce(r32.grad, op=dist.ReduceOp.AVG)   # the path's one exchange step: NCCL mean over NVLink
                else:
                    r32.grad.div_(world)             # with the peer ring the backward already returned the sum
            if keep is not None:
                keep.update(("grad_" + k, t[k].grad) for k in ROW_KEYS if k != "y")
                keep["grad_r_sqrt_sigma"] = r32.grad
            for k in ROW_KEYS:
                if k != "y":
                    t[k].grad = None
                    t[k].requires_grad_(False)
        if from_host:
            # the step's result as train.py:131 consumes it: the loss and the eight batch metrics (computed on the
            # device, SURVEY 8f-N1: mpvae_b200.metrics.batch_metrics) come back to the host
            metrics_host.copy_(batch_metrics_tensor(out[6], t["y"], 0.5), non_blocking=True)
            loss_host.copy_(out[0].detach(), non_blocking=True)
        if keep is not None:
            keep.update(zip(OUT_NAMES, out))
        return out

    def timed_e2e(leg, n_steps):
        """K steps through the public API starting from pinned HOST buffers: every step's inputs cross PCIe inside the
        timed region (double-buffered on a side stream by mpvae_b200.train.HostBatchPrefetcher) and the loss + metrics
        come back to the host.  One event pair around all K steps; the working set is far larger than L2."""
        from mpvae_b200.train import HostBatchPrefetcher
        pf = HostBatchPrefetcher(dev, depth=2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pf.push(leg.host)
        for i in range(n_steps):
            batch = pf.next()
            if i + 1 < n_steps:
                pf.push(leg.host)
            one_step(leg, batch, True)
            pf.release()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def timed(leg, n_steps, keep=None, **kw):
        evs = []
        for i in range(n_steps):
            flush.add_(1.0)                         # evict L2 between timed iterations (2 x 126 MB written)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one_step(leg, leg.dev, False, keep=keep if i == n_steps - 1 else None, **kw)
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return [e0.elapsed_time(e1) for e0, e1 in evs]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        if world == 1:
            return list(vals)
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    warm = max(3, a.warmup)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()             # started ahead of the warm-up: its first sample takes a few hundred ms
    for _ in range(warm):
        one_step(main, main.dev, False)
    timed_e2e(main, 2)
    barrier()
    sampler.mark_begin()            # clocks are reported for the two timed regions below only
    launches0 = _lib.launch_count()
    last = {} if a.dump_outputs else None
    ms = timed(main, a.steps, keep=last)
    launches = _lib.launch_count() - launches0
    if last is not None and rank == 0:
        # before any further step: with the peer ring, g_R lives in the ring's buffer, which the next step overwrites
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in host_outputs(last).items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    last = None
    barrier()
    total_ms = sum(ms)
    total_e2e = timed_e2e(main, a.steps)
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    total_ms, total_e2e = max_over_ranks(total_ms, total_e2e)
    if a.profile_host and world == 1:      # (one process only: under N ranks a lone rank would wait for the others' exchange)
        import cProfile
        import io
        import pstats
        torch.cuda.synchronize()
        prof = cProfile.Profile()
        t0 = time.perf_counter()
        prof.enable()
        timed_e2e(main, 20)
        prof.disable()
        buf = io.StringIO()
        pstats.Stats(prof, stream=buf).sort_stats("cumulative").print_stats(45)
        print(f"[bench] host wall per e2e step (incl. the final sync): {(time.perf_counter() - t0) / 20 * 1e3:.3f} ms\n"
              + buf.getvalue(), file=sys.stderr)
    if ring is not None:
        ring.check()                # a flag wait that timed out would have produced invalid sums

    # ---- N > 1: the exchange checked against NCCL, and the other scaling mode as a short leg ----
    exchange_check = None
    other_leg = None
    if world > 1 and not infer:
        if ring is not None:
            # one untimed step twice with the same noise: g_R over the peer ring vs NCCL's all-reduce of the partials
            step_no[0] = 10_000
            one_step(main, main.dev, False, use_ring=True)
            g_ring = r32.grad.detach().clone()
            step_no[0] = 10_000
            one_step(main, main.dev, False, use_ring=False)
            g_nccl = r32.grad.detach()
            diff = (g_ring - g_nccl).abs().max() / g_nccl.abs().max().clamp_min(1e-30)
            dist.all_reduce(diff, op=dist.ReduceOp.MAX)
            exchange_check = {"max_rel_diff_vs_nccl_allreduce": float(diff), "ok": bool(float(diff) <= 2e-6)}
        other = "strong" if a.scaling == "weak" else "weak"
        if other == "strong":
            lo, hi = shard_rows(B, rank, world)
            leg2 = Leg(B, lo, hi, 300 + rank) if hi > lo else None
        else:
            leg2 = Leg(B * world, rank * B, (rank + 1) * B, 300 + rank)
        have = torch.tensor([1 if leg2 is not None else 0], device=dev)
        dist.all_reduce(have, op=dist.ReduceOp.MIN)
        if int(have.item()):
            k2 = max(3, min(a.steps, 20))
            for _ in range(3):
                one_step(leg2, leg2.dev, False)
            barrier()
            (t2,) = max_over_ranks(sum(timed(leg2, k2)))
            barrier()
            other_leg = {"scaling": other, "B_global": leg2.Bg, "rows_this_rank": leg2.hi - leg2.lo, "steps": k2,
                         "ms_per_step": t2 / k2, "value": float(S) * leg2.Bg * L * k2 / (t2 * 1e-3), "unit": UNIT}

    # ---- per-kernel device times inside the step (library CUDA-event records) -> roofline of the dominant kernel ----
    roof = None
    Bl = main.hi - main.lo
    cells = float(S) * Bl * L
    kp = max(3, min(a.steps, 10))
    _lib.profile(True)
    timed(main, kp)
    prof = _lib.profile_read()
    _lib.profile(False)
    kernels = {k: v[0] / v[1] for k, v in prof.items()}
    barrier()
    kernels_by_rank = None
    if world > 1:
        # every rank's per-kernel times: the spread over the ranks of a kernel that WAITS for the others (the exchange, and
        # the g_R product when the exchange runs beside it) is the skew, the spread of the others is rank-to-rank variation
        gathered = [None] * world
        dist.all_gather_object(gathered, kernels)
        keys = list(kernels)
        kernels_by_rank = {k: {"min": min(g.get(k, float("nan")) for g in gathered),
                               "max": max(g.get(k, float("nan")) for g in gathered),
                               "ranks": [round(g.get(k, float("nan")), 4) for g in gathered]} for k in keys}
        kernels_by_rank["sum of the kernels"] = {"ranks": [round(sum(g.values()), 4) for g in gathered]}
    if rank == 0:
        f_max = peaks["sm_max_mhz"] * 1e6
        nt_key = next((k for k in kernels if k.startswith("product nt")), None)
        top = max(kernels, key=kernels.get)
        if dense and nt_key:
            t_k = kernels[nt_key] * 1e-3
            # algorithmic flops of the launch (cost model v0): the contraction, plus the forward cell work it carries
            flops = cells * (2.0 * Z + (120.0 if fused else 0.0))
            peak = peaks["bf16_tflops"] / passes
            roof = {"bound": "tensor", "achieved": flops / t_k / 1e12, "peak": peak, "unit": "TFLOP/s",
                    "frac": flops / t_k / 1e12 / peak,
                    "traffic": TRAFFIC.get((L, Z, S * Bl, bool(fused))),
                    "kernel": "gemm_split_2sm_kernel<nt> (noise.R^T, mpvae.py:168" + (" + the row forward :177-204 on its math warps" if fused
                                                                                   else " + the Philox draw of mpvae.py:162 on its math warps")
                              + f"), tcgen05 fp16 hi/lo split, {passes} MMA passes",
                    "kernel_ms": t_k * 1e3, "timed": "CUDA events recorded by the library around the launch, inside the step",
                    "peak_basis": f"{peaks['_source']} bf16 burst {peaks['bf16_tflops']} TFLOP/s / {passes} "
                                  f"(fp32-equivalent flops of a {passes}-pass split-precision product)",
                    "frac_of_sustained": flops / t_k / 1e12 / (peaks["bf16_tflops_sustained"] / passes),
                    "algorithmic_flops_per_launch": flops}
        else:
            # CUDA-core regime (SURVEY 8d regime (i)): the dominant kernel against the FP32 issue rate
            t_k = kernels[top] * 1e-3
            per_cell = {"row forward": 120.0, "row backward": 80.0, "product nt": 2.0 * Z, "product tn": 2.0 * Z,
                        "fused small-regime forward": 2.0 * Z + 120.0, "fused small-regime backward": 2.0 * Z + 80.0}
            fl = next((v for k, v in per_cell.items() if top.startswith(k)), 120.0) * cells
            peak = FP32_LANES * f_max / 1e12
            roof = {"bound": "fp32", "achieved": fl / t_k / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": fl / t_k / 1e12 / peak,
                    "traffic": None, "kernel": top, "kernel_ms": t_k * 1e3,
                    "timed": "CUDA events recorded by the library around the launch, inside the step",
                    "peak_basis": f"148 SMs x 128 FMA lanes x 2 x {peaks['sm_max_mhz']:.0f} MHz (CUDA-core FP32 issue, SURVEY 8d regime (i))",
                    "algorithmic_flops_per_launch": fl}
        cm = cost_model(S, Bl, L, Z, D, not infer, dense, passes, peaks)
        roof["step_frac"] = cm["t_min_ms"] / (total_ms / a.steps)
        roof["step_model"] = cm

    # ---- the same loss step captured ONCE as a CUDA graph and replayed (no host work between the launches), N = 1 ----
    graph_leg = None
    if world == 1 and total_ms / a.steps < 0.5:      # launch-bound workloads only: a dense step gains nothing from a graph
        try:
            import copy
            gargs = copy.copy(main.args)
            gargs.noise_offset_tensor = torch.zeros(1, dtype=torch.int64, device=dev)   # Philox offset bumped inside the graph
            gargs.noise_offset = 0
            gargs.peer_ring = None
            g_leaves = {k: (main.dev[k] if k == "y" else main.dev[k].detach().clone().requires_grad_(not infer)) for k in ROW_KEYS}
            g_r32 = r32.detach().clone().requires_grad_(not infer)

            def graph_body():
                with torch.no_grad() if infer else torch.enable_grad():
                    out = M.compute_loss(g_leaves["y"], g_leaves["fe_out"], g_leaves["fe_mu"], g_leaves["fe_logvar"],
                                         g_leaves["fx_out"], g_leaves["fx_mu"], g_leaves["fx_logvar"], g_r32, gargs)
                    if not infer:
                        out[0].backward()
                gargs.noise_offset_tensor.add_(1)
                return out

            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    for t in list(g_leaves.values()) + [g_r32]:
                        t.grad = None
                    graph_body()
            torch.cuda.current_stream(dev).wait_stream(side)
            for t in list(g_leaves.values()) + [g_r32]:
                t.grad = None
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                g_out = graph_body()
            for _ in range(3):
                graph.replay()
            evs = []
            for _ in range(a.steps):
                flush.add_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); graph.replay(); e1.record()
                evs.append((e0, e1))
            torch.cuda.synchronize()
            g_ms = sum(e0.elapsed_time(e1) for e0, e1 in evs) / a.steps
            graph_leg = {"ms_per_step": g_ms, "value": float(S) * Bl * L / (g_ms * 1e-3), "unit": UNIT, "loss": float(g_out[0].detach()),
                         "what": "the same Philox draw + forward + backward as `value`, captured once as a CUDA graph and replayed "
                                 "(device-side Philox offset); L2 flushed between replays"}
            del graph
        except Exception as exc:   # noqa: BLE001 -- informative leg
            graph_leg = {"error": repr(exc)[:200]}

    # ---- the three-pass route (external fp32 noise tensor, e.g. args.noise_mode = 'reference'), N = 1 ----
    ext_ms = None
    if world == 1 and dense and not infer:
        nz = torch.randn(S, Bl, Z, device=dev)
        for _ in range(2):
            one_step(main, main.dev, False, noise=nz)
        ke = max(3, min(a.steps, 10))
        ext_ms = sum(timed(main, ke, noise=nz)) / ke
        del nz

    # ---- full training step (train.py:103-129: VAE fwd -> loss -> bwd -> all-reduce -> clip -> Adam -> StepLR) ----
    train = None
    if not a.no_train_step and not infer:
        from types import SimpleNamespace
        from mpvae_b200.train import DataParallelStep
        Bg = main.Bg
        margs = SimpleNamespace(feature_dim=sh.feature_dim, label_dim=L, latent_dim=D, z_dim=Z, keep_prob=0.5,
                                scale_coeff=1.0, residue_sigma="", n_train_sample=S, n_test_sample=S, mode="train",
                                nll_coeff=0.5, c_coeff=10.0, mpvae_flags=flags, noise_seed=99)
        np.random.seed(4)
        torch.manual_seed(0)
        vae = M.VAE(margs).to(dev)
        from mpvae_b200.optim import FusedAdam
        opt = FusedAdam(vae.parameters(), lr=torch.tensor(1e-3, device=dev), weight_decay=1e-5)
        sched = torch.optim.lr_scheduler.StepLR(opt, 1000, 0.5)
        stepper = DataParallelStep(vae, opt, sched, margs, clip_norm=100.0)
        rng = np.random.RandomState(5)
        xg = torch.from_numpy(synth.features(Bg, sh.feature_dim, rng)).to(dev)
        yg = torch.from_numpy(synth.labels(Bg, L, sh.label_rate, rng)).to(dev)
        k_train = max(3, min(a.steps, 20))

        def time_steps(fn):
            for _ in range(3):
                fn(yg, xg)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_wall = time.perf_counter()
            e0.record()
            for _ in range(k_train):
                out = fn(yg, xg)
            e1.record()
            torch.cuda.synchronize()
            t_wall = time.perf_counter() - t_wall
            (t_dev,) = max_over_ranks(e0.elapsed_time(e1))
            return t_dev / k_train, t_wall * 1e3 / k_train, out

        eager_ms, eager_wall, out_t = time_steps(stepper.step)
        train = {"steps_per_s": 1e3 / eager_ms, "ms_per_step": eager_ms, "wall_ms_per_step": eager_wall,
                 "steps": k_train, "global_batch": Bg, "params": int(sum(p.numel() for p in vae.parameters())),
                 "loss": float(out_t.total_loss.detach()),
                 "what": "zero_grad, VAE fwd (large layers on this library's tcgen05 engine), probit ELBO fwd+bwd (this library), "
                         "MLP bwd, grad all-reduce, clip_grad_norm_(100) + Adam(wd=1e-5) (mpvae_b200.optim.FusedAdam), "
                         "StepLR; per-step host metrics excluded"}
        from mpvae_b200.train import GraphedTrainStep
        if world > 1:
            # the NCCL-free step: g_R summed beside its product, the rest of the gradient bucket (and the loss terms) in
            # place over NVLink peer memory by the library's exchange kernel -- and, because no NCCL call is left, the
            # whole N-rank step as a CUDA graph.  Set-up is collective; a failure on any rank is reported, not fatal.
            vae = opt = stepper = None
            try:
                np.random.seed(4)
                torch.manual_seed(0)
                vae = M.VAE(margs).to(dev)
                opt = FusedAdam(vae.parameters(), lr=torch.tensor(1e-3, device=dev), weight_decay=1e-5)
                sched = torch.optim.lr_scheduler.StepLR(opt, 1000, 0.5)
                stepper = DataParallelStep(vae, opt, sched, margs, clip_norm=100.0, peer_g_r=True, peer_all=True)
                if stepper.pbucket is None:
                    raise RuntimeError("peer-mapped gradient bucket unavailable")
                p_ms, p_wall, out_p = time_steps(stepper.step)
                train["nccl_free"] = {"steps_per_s": 1e3 / p_ms, "ms_per_step": p_ms, "wall_ms_per_step": p_wall,
                                      "loss": float(out_p.total_loss.detach()),
                                      "what": "DataParallelStep(peer_g_r=True, peer_all=True): no NCCL call in the step"}
            except Exception as exc:   # noqa: BLE001
                train["nccl_free"] = {"error": repr(exc)[:200]}
                stepper = None
        try:   # the same step captured once as a CUDA graph and replayed (mpvae_b200.train.GraphedTrainStep)
            if stepper is None:
                raise RuntimeError("no stepper to capture")
            graphed = GraphedTrainStep(stepper)
            g_ms, g_wall, out_g = time_steps(graphed.step)
            train["cuda_graph"] = {"steps_per_s": 1e3 / g_ms, "ms_per_step": g_ms, "wall_ms_per_step": g_wall,
                                   "loss": float(out_g.total_loss.detach())}
            if world > 1:
                train["cuda_graph"]["what"] = "the NCCL-free step captured on every rank"
                for r_ in (stepper.ring, stepper.pbucket):
                    if r_ is not None:
                        r_.check()
        except Exception as exc:   # noqa: BLE001 - the graph leg is informative, never fatal for the bench line
            train["cuda_graph"] = {"error": repr(exc)[:200]}
        vae = opt = stepper = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    Bg = main.Bg
    units = float(S) * Bg * L * a.steps
    bi = sum(main.host[k].numel() * main.host[k].element_size() for k in ROW_KEYS)
    line = {
        "metric": METRIC, "value": units / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": warm, "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": a.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "dtype_note": "fp32 arithmetic and fp32-accurate products (fp16 hi/lo split-precision tensor-core passes accumulated in fp32); "
                      "the library's own Philox normals are DEFINED on the fp16 grid (a changed input distribution, not a reduced "
                      "compute precision); external_noise_ms_per_step is the same step fed arbitrary fp32 noise",
        "config": {"workload": f"{sh.name}-shaped S{S} B{B} L{L} Z{Z} " + ("inference (forward, no_grad)" if infer else "fwd+bwd"),
                   "S": S, "B_per_gpu": Bl, "B_global": Bg, "L": L, "Z": Z, "D": D,
                   "noise": "philox, drawn by the library inside the step on the fp16 grid (fp32 arithmetic everywhere else; an "
                            "external fp32 noise tensor takes three MMA passes instead of two: external_noise_ms_per_step)",
                   "engine": a.engine, "row_forward": ("fused into the product kernel" if fused else "separate kernel"),
                   "l2": "L2 flushed between timed iterations (252 MB written); per-step CUDA events summed",
                   "exchange": ("none (1 GPU)" if world == 1 else
                                ("g_R summed inside the NVSwitch (multimem.ld_reduce / multimem.st by the chunk owners), inside "
                                 "the backward") if (ring is not None and a.exchange == "nvls") else
                                ("g_R summed over NVLink peer memory after the product (chunk owners pull, add in rank order, "
                                 "store to every rank)" if a.serial_exchange else
                                 "g_R summed over NVLink peer memory slab by slab BESIDE the g_R product: the product leaves 8 SMs "
                                 "free and publishes finished tiles; an exchange kernel on those SMs pulls each finished 256-row "
                                 "slab from every rank, adds in rank order, stores to every rank; the K-sliced tail rows after the "
                                 "product" if not a.fused_exchange else
                                 "g_R summed over NVLink peer memory INSIDE the g_R product kernel, tile by tile (tile t belongs to "
                                 "rank t mod N: its math warps pull the finished tile from every rank, add in rank order, store to "
                                 "every rank; the K-sliced tail rows by the stand-alone reduce kernel)") if ring is not None
                                else "NCCL all-reduce of g_R (fp32) per step")},
        "clocks": clocks,
        "e2e": {"value": units / (total_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": bi, "d2h_bytes_per_step": 4 + 64,
                "how": "mpvae_b200.compute_loss + backward from pinned host buffers (labels as bits: mpvae_b200.train.pack_labels, the rest fp32), H2D "
                       "double-buffered on a side stream; the loss and the step's eight metrics (train.py:131, computed on "
                       "the device by mpvae_b200.metrics.batch_metrics) copied back to the host every step",
                "ms_per_step": total_e2e / a.steps},
        "gpu_launches": int(launches),
        "loss_steps_per_s": a.steps / (total_ms * 1e-3),
        "kernel_ms": kernels, "kernel_ms_by_rank": kernels_by_rank,
        "train_step": train,
        "roofline": roof,
    }
    if exchange_check is not None:
        line["exchange_check"] = exchange_check
    if other_leg is not None:
        line[other_leg["scaling"] + "_scaling"] = other_leg
    if ext_ms is not None:
        line["external_noise_ms_per_step"] = ext_ms
    if graph_leg is not None:
        line["cuda_graph_loss_step"] = graph_leg
        if "ms_per_step" in graph_leg and roof is not None:
            roof["step_frac_cuda_graph"] = roof["step_model"]["t_min_ms"] / graph_leg["ms_per_step"]
    ref = None
    if not (a.no_cpu_baseline and a.no_torch_baseline):
        ref = _reference_module()
    if world == 1 and not a.no_torch_baseline:
        # what a user of the reference's train.py:20 (cuda:0) sees on this same B200: stock torch CUDA ops.  The
        # unmodified compute_loss where its O(L^2) ranking loss fits in memory, else the oracle port's exact
        # factorisation of that loss (the only way eurlex fits anywhere).
        try:
            pair_bytes = 6.0 * S * Bl * L * L * 4
            if ref is not None and pair_bytes < 60e9:
                fn = lambda i: cpu_reference_step(L, Z, S, Bl, seed=i, device=dev, ref=ref, train=not infer)   # noqa: E731
                what = "unmodified /root/reference/mpvae.py compute_loss (oracle/_ref/) with CUDA tensors"
                kind = "reference"
            else:
                fn = lambda i: torch_factorised_step(L, Z, S, Bl, i, dev, not infer)   # noqa: E731
                what = "oracle port with the ranking loss factorised (the pairwise form needs %.0f GB), torch CUDA ops" % (pair_bytes / 1e9)
                kind = "port-factorised"
            for i in range(3):
                fn(i)
            tt = [fn(10 + i) for i in range(5)]
            t_ref = statistics.median(tt)
            line["torch_cuda_baseline"] = {"value": cells / t_ref, "unit": UNIT, "ms_per_step": t_ref * 1e3, "kind": kind,
                                           "what": what + (", fwd+bwd" if not infer else ", forward") +
                                                   "; wall clock with device sync, inputs resident, its own noise draw (host) included",
                                           "speedup_of_value": (units / (total_ms * 1e-3)) / (cells / t_ref)}
        except Exception as exc:   # noqa: BLE001 -- informative leg
            line["torch_cuda_baseline"] = {"error": repr(exc)[:200]}
        torch.cuda.empty_cache()
    if not a.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count())
        kind, what = cpu_kind(ref)
        rows = cpu_rows_for(L, Z, S, Bl, a.cpu_rows)
        cpu_reference_step(L, Z, S, min(rows, 1), ref=ref, train=not infer)
        t_cpu = cpu_reference_step(L, Z, S, rows, ref=ref, train=not infer)
        line["cpu_baseline"] = {"value": S * rows * L / t_cpu, "unit": UNIT, "cores": torch.get_num_threads(),
                                "kind": kind,
                                "sample": f"1 step on {rows} of {Bl} rows ({t_cpu:.1f} s): {what} "
                                          "(O(L^2) pairwise ranking loss) on torch CPU, " + ("fwd+bwd" if not infer else "forward")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
