#!/usr/bin/env python
"""Fiat-Shamir over packed records against the byte-plane Fiat-Shamir calls, per 2^20 items, one process.

1. Kernel times (CUDA events on the context's stream, warm-up first, 20 launches per figure): pbh_prove_fs_batch_dev /
   pbh_verify_fs_batch_dev against pbh_prove_fs_packed_dev / pbh_verify_fs_packed_dev, PBH_ALGO_TABLE and PBH_ALGO_ARITH, on
   D_uniform witnesses and on the batch in which every item completes the transcript (scripts/time_fs.py builds the same one).
2. End to end, 2^20 prove + verify pairs from host memory (host clock around calls that return after their last copy; median
   of 7 after 2 warm-up passes): byte-plane synchronous calls on page-locked memory, packed synchronous calls, packed calls on
   four lanes over host_alloc_as buffers.  No challenge outputs are requested in this part (a caller that only proves and
   verifies needs none): 21 B up / 28 B down per proof and 27 B up / 1 B down per verification for byte planes, 12 / 12 and
   12 / 1 for packed records.
Every output is compared with the byte-plane result of the same inputs.  The card's name and power limit are read in the same
run and printed first."""
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "plonk-by-fingers_b200", "python"))
import numpy as np
import torch
import pbh_b200 as P

n = 1 << 20
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi.stdout.strip() or smi.stderr.strip()}")
ctx = P.Context(device=0)
stream = ctx.torch_stream()
dev = torch.device("cuda", 0)


def timed(fn, reps=20):
    with torch.cuda.stream(stream):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3     # us per call


def host_timed(fn, reps=7):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts) * 1e6          # us per call


def line(what, t_plane, t_packed):
    print(f"  {what:<58s} planes {t_plane:8.1f} us   packed {t_packed:8.1f} us   packed / planes {t_packed / t_plane:6.3f}")


# ---- 1. kernels --------------------------------------------------------------------------------------------------------------
w, r, _, _ = ctx.generate_inputs(n, seed=1, dist=P.DIST_UNIFORM)
proof = torch.empty((27, n), dtype=torch.uint8, device=dev); status = torch.empty((n,), dtype=torch.uint8, device=dev)
chal = torch.empty((6, n), dtype=torch.uint8, device=dev); result = torch.empty((n,), dtype=torch.uint8, device=dev)
pout = torch.empty((12 * n,), dtype=torch.uint8, device=dev); pcu = torch.empty((4 * n,), dtype=torch.uint8, device=dev)
pres = torch.empty((n,), dtype=torch.uint8, device=dev)
ctx.prove_fs_batch(w, r, proof=proof, status=status, want_chal=False)
ctx.sync()
idx = torch.nonzero(status == 0).flatten()
idx = idx.repeat((n + idx.numel() - 1) // idx.numel())[:n]
batches = {"D_uniform": (w, r), "all items complete": (w[:, idx].contiguous(), r[:, idx].contiguous())}
print(f"kernels, {n} items, CUDA events, 20 launches after 3 warm-up launches")
for algo in ("table", "arith"):
    ctx.set_algo(algo)
    for bname, (bw, br) in batches.items():
        pin = torch.from_numpy(P.pack_fs_witness(bw.cpu().numpy(), br.cpu().numpy()).view(np.uint8)).to(dev)
        # same bytes first
        ctx.prove_fs_batch(bw, br, proof=proof, status=status, chal=chal)
        ctx.verify_fs_batch(proof, result=result, want_chal=False)
        ctx.prove_fs_packed(pin, out=pout, chal_u=pcu)
        ctx.verify_fs_packed(pout, result=pres)
        ctx.sync()
        pk = pout.cpu().numpy().view(P.PACKED_PROOF)
        assert np.array_equal(pk, P.pack_proofs(proof.cpu().numpy(), status.cpu().numpy())), (algo, bname)
        c = chal.cpu().numpy()
        assert np.array_equal(pcu.cpu().numpy().view("<u4"), P.pack_chal_u(c[:5], c[5])), (algo, bname)
        assert torch.equal(pres, result), (algo, bname)
        done = float((status == 0).float().mean())
        print(f"[{algo}] {bname} ({100 * done:.1f} % of the proofs complete)")
        line("prove, challenges returned (5 compressions)",
             timed(lambda: ctx.prove_fs_batch(bw, br, proof=proof, status=status, chal=chal)),
             timed(lambda: ctx.prove_fs_packed(pin, out=pout, chal_u=pcu)))
        line("prove, challenges not returned (u not derived)",
             timed(lambda: ctx.prove_fs_batch(bw, br, proof=proof, status=status, want_chal=False)),
             timed(lambda: ctx.prove_fs_packed(pin, out=pout, want_chal_u=False)))
        line("verify of those proofs",
             timed(lambda: ctx.verify_fs_batch(proof, result=result, want_chal=False)),
             timed(lambda: ctx.verify_fs_packed(pout, result=pres)))
ctx.set_algo("table")

# ---- 2. end to end -----------------------------------------------------------------------------------------------------------
bw, br = (t.cpu().numpy() for t in batches["D_uniform"])
print(f"end to end, {n} prove + verify pairs from host memory, PBH_ALGO_TABLE, D_uniform witnesses, host clock, median of 7")
hw, hr, hp, hs, hres = (ctx.host_alloc((k, n)) for k in (12, 9, 27, 1, 1))
hw[...] = bw; hr[...] = br
ref_p, ref_s = ctx.prove_fs_batch(bw, br, want_chal=False)
ref_v = ctx.verify_fs_batch(ref_p, want_chal=False)
ref_pk = P.pack_proofs(ref_p, ref_s)


def planes_sync():
    ctx.prove_fs_batch(hw, hr, proof=hp, status=hs[0], want_chal=False)
    ctx.verify_fs_batch(hp, result=hres[0], want_chal=False)


t_planes = host_timed(planes_sync)
assert np.array_equal(hp, ref_p) and np.array_equal(hres[0], ref_v)
pin_h = ctx.host_alloc_as(n, P.PACKED_FS_WITNESS); pout_h = ctx.host_alloc_as(n, P.PACKED_PROOF); pres_h = ctx.host_alloc_as(n, np.uint8)
pin_h[...] = P.pack_fs_witness(bw, br)


def packed_sync():
    ctx.prove_fs_packed(pin_h, out=pout_h, want_chal_u=False)
    ctx.verify_fs_packed(pout_h, result=pres_h)


t_packed = host_timed(packed_sync)
assert np.array_equal(pout_h, ref_pk) and np.array_equal(pres_h, ref_v)
q = n // 4


def packed_lanes():
    for lane in range(4):
        s = slice(lane * q, (lane + 1) * q)
        ctx.prove_fs_packed_async(lane, pin_h[s], pout_h[s])
        ctx.verify_fs_packed_async(lane, pout_h[s], pres_h[s])
    ctx.sync()


pout_h.view(np.uint8)[...] = 0; pres_h[...] = 0xEE
t_lanes = host_timed(packed_lanes)
assert np.array_equal(pout_h, ref_pk) and np.array_equal(pres_h, ref_v)
for name, t in (("byte planes, synchronous calls, page-locked", t_planes), ("packed records, synchronous calls, page-locked", t_packed),
                ("packed records, four lanes of 2^18, host_alloc_as buffers", t_lanes)):
    print(f"  {name:<58s} {t:9.1f} us   {n / t / 1e3:6.3f} G pairs/s")
for a in (hw, hr, hp, hs, hres, pin_h, pout_h, pres_h):
    ctx.host_free(a)
ctx.close()
