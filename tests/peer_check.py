"""2+ GPU check (not a pytest test; run under torchrun): g_R summed over ranks inside the probit backward through NVLink
peer memory (mpvae_b200.peer.PeerRing) against the NCCL all-reduce of the per-rank g_R.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/peer_check.py
"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from mpvae_b200 import synth
from mpvae_b200.mpvae import compute_loss
from mpvae_b200.peer import NvlsRing, PeerRing


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    # the exchange runs BESIDE the g_R product from S * B >= 8192 rows per rank (all full slabs published; 7 of 9 slabs + a
    # K-sliced tail; ragged Z), behind it below that and when every tile is K-sliced (1000 x 700: twelve tiles)
    for (L, Z, B, S) in ((983, 983, 128, 10), (3993, 3993, 512, 10), (3993, 3993, 1024, 10), (2304, 2100, 1024, 8),
                         (1000, 700, 1024, 10)):
        inp = synth.loss_inputs(L, Z, B * world, S, seed=11, with_noise=False, label_rate=20.0 / L)
        rows = slice(rank * B, (rank + 1) * B)
        t = {k: torch.from_numpy(v if k == "r_sqrt_sigma" else v[rows]).to(dev) for k, v in inp.items()}
        # PEER_CHECK_RING=nvls: the in-switch reduction (multimem) instead of the pull kernel
        ring = (NvlsRing if os.environ.get("PEER_CHECK_RING") == "nvls" else PeerRing)(L, Z, dev)

        def run(use_ring, step):
            # PEER_CHECK_SERIAL=1: the sum runs after the g_R product at every shape (MPVAE_FLAG_SERIAL_EXCHANGE)
            args = synth.make_args(L, Z, n_train_sample=S, noise_seed=5, noise_offset=step,
                                   mpvae_flags=(0x80 if os.environ.get("PEER_CHECK_SERIAL") == "1" else 0) if use_ring else 0)
            args.dp_global_batch, args.dp_row0 = B * world, rank * B
            args.peer_ring = ring if use_ring else None
            leaves = {k: (v if k in ("y", "r_sqrt_sigma") else v.clone().requires_grad_(True)) for k, v in t.items()}
            r32 = t["r_sqrt_sigma"].float().requires_grad_(True)
            out = compute_loss(leaves["y"], leaves["fe_out"], leaves["fe_mu"], leaves["fe_logvar"], leaves["fx_out"],
                               leaves["fx_mu"], leaves["fx_logvar"], r32, args)
            out[0].backward()
            g = r32.grad.clone()
            if not use_ring:
                dist.all_reduce(g)
            return g

        for step in range(4):                                  # several steps: the buffers are reused
            g_ring, g_nccl = run(True, step), run(False, step)
            rel = ((g_ring - g_nccl).abs().max() / g_nccl.abs().max()).item()
            gathered = [torch.empty_like(g_ring) for _ in range(world)]
            dist.all_gather(gathered, g_ring)
            same = all(torch.equal(gathered[0], x) for x in gathered)
            if rank == 0:
                print(f"L={L} Z={Z} B/rank={B} step {step}: ring vs nccl rel diff {rel:.2e}, identical on all ranks: {same}")
            ok = ok and rel <= 2e-6 and same

        def timed(use_ring, n=10):
            for i in range(3):
                run(use_ring, 100 + i)
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                run(use_ring, 200 + i)
            e1.record(); torch.cuda.synchronize()
            tt = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return tt.item()

        # the exchange alone: library all-reduce over peer memory vs NCCL, same 4*L*Z bytes
        def time_x(fn, n=20):
            for _ in range(3):
                fn()
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record(); torch.cuda.synchronize()
            tt = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return tt.item()
        ring.part.normal_()
        buf = ring.part.clone()
        want = buf.clone(); dist.all_reduce(want)
        got = ring.allreduce()
        x_ok = bool(((got - want).abs().max() / want.abs().max()) < 1e-6)
        gathered = [torch.empty_like(got) for _ in range(world)]
        dist.all_gather(gathered, got.contiguous())
        x_ok = x_ok and all(torch.equal(gathered[0], t_) for t_ in gathered)
        t_x_ring, t_x_nccl = time_x(ring.allreduce), time_x(lambda: dist.all_reduce(buf))
        if rank == 0:
            print(f"L={L}: exchange alone ({4 * L * Z / 1e6:.0f} MB): peer {t_x_ring * 1e3:.0f} us, nccl {t_x_nccl * 1e3:.0f} us, equal: {x_ok}")
        ok = ok and x_ok
        t_ring, t_nccl = timed(True), timed(False)
        if rank == 0:
            print(f"L={L}: loss fwd+bwd+exchange per step: peer ring {t_ring:.3f} ms, nccl {t_nccl:.3f} ms")
        ring.close()
    # the gradient bucket of the NCCL-free step: ranges of one peer-mapped buffer summed in place
    from mpvae_b200.peer import PeerBucket
    n = 3_000_011
    bucket = PeerBucket(n, dev)
    for first, cnt in ((0, n), (1024, n - 1024), (4, 1001), (n - 7 - (n - 7) % 4, None)):
        bucket.flat.normal_()
        want = bucket.flat.clone()
        lo_, hi_ = first, n if cnt is None else first + cnt
        seg = want[lo_:hi_].clone(); dist.all_reduce(seg); want[lo_:hi_] = seg
        torch.cuda.synchronize(); dist.barrier()          # every rank has filled its buffer before anyone pulls
        got = bucket.allreduce(first, cnt).clone()
        rel = ((got - want).abs().max() / want.abs().max()).item()
        gathered = [torch.empty_like(seg) for _ in range(world)]
        dist.all_gather(gathered, got[lo_:hi_].contiguous())
        same = all(torch.equal(gathered[0], x) for x in gathered)
        if rank == 0:
            print(f"bucket [{lo_}, {hi_}) in place: rel diff vs nccl {rel:.2e}, range identical on all ranks: {same}")
        ok = ok and rel <= 1e-6 and same
    bucket.check()
    bucket.close()
    if rank == 0:
        print("PEER_CHECK", "PASS" if ok else "FAIL")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
