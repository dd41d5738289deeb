#!/usr/bin/env python
"""Fiat-Shamir shard summaries: fused against unfused, and the Fiat-Shamir sharded pass, in one process.

1. Kernel times (CUDA events on the context's stream), 2^20 and 2^24 items of D_fullpath witnesses, PBH_ALGO_TABLE and
   PBH_ALGO_ARITH: the Fiat-Shamir prover alone (pbh_prove_fs_batch_dev, no challenge planes), the prover followed by
   pbh_digest_dev (unfused), and pbh_prove_fs_digest_batch_dev (fused); the same three for the verifier and the verdict bitmap
   (pbh_verify_fs_batch_dev, + pbh_pack_verdicts_dev, pbh_verify_fs_bitmap_batch_dev).  The three variants of a row are timed
   in alternation, five rounds of 20 (2^20) or 3 (2^24) launches after warm-up; each figure is the median round.
2. pbh_multi_prove_verify_fs_sharded with 2^24 items per device (weak scaling) on one device and on every visible device: median of
   7 passes after 2 warm-up passes, device time of the pass including the all-gather (CUDA events inside the library).
Every fused output is compared with the unfused one before it is timed.  The card's name, power limit and SM clock are read in
the same run and printed first.  Usage: time_fs_sharded.py [--out FILE] (default profiles/r05a_fs_sharded.txt)."""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "plonk-by-fingers_b200", "python"))
import torch
import pbh_b200 as P

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05a_fs_sharded.txt"))
args = ap.parse_args()
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True)
say(f"device: {torch.cuda.get_device_name(0)}; visible devices: {torch.cuda.device_count()}")
say(f"nvidia-smi name, power limit, SM clock, max SM clock: {smi.stdout.strip() or smi.stderr.strip()}")
ctx = P.Context(device=0)
stream = ctx.torch_stream()
dev = torch.device("cuda", 0)


def rounds(fns, reps, n_rounds=5):
    """Median over rounds of the mean time per launch (us) of each fn, the fns alternating within a round."""
    out = [[] for _ in fns]
    with torch.cuda.stream(stream):
        for fn in fns:
            for _ in range(2):
                fn()
        for _ in range(n_rounds):
            for k, fn in enumerate(fns):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(reps):
                    fn()
                e1.record(stream)
                e1.synchronize()
                out[k].append(e0.elapsed_time(e1) / reps * 1e3)
    return [statistics.median(t) for t in out]


say("1. kernels, D_fullpath witnesses, CUDA events, median of 5 alternating rounds")
for n in (1 << 20, 1 << 24):
    reps = 20 if n == 1 << 20 else 3
    w, r, _, _ = ctx.generate_inputs(n, seed=0xB200, dist=P.DIST_FULLPATH)
    proof = torch.empty((27, n), dtype=torch.uint8, device=dev); status = torch.empty((n,), dtype=torch.uint8, device=dev)
    result = torch.empty((n,), dtype=torch.uint8, device=dev); bitmap = torch.empty((n // 8,), dtype=torch.uint8, device=dev)
    dg = torch.empty((1,), dtype=torch.int64, device=dev); dg2 = torch.empty((1,), dtype=torch.int64, device=dev)
    bm2 = torch.empty((n // 8,), dtype=torch.uint8, device=dev)
    for algo in ("table", "arith"):
        ctx.set_algo(algo)
        with torch.cuda.stream(stream):
            ctx.prove_fs_batch(w, r, proof=proof, status=status, want_chal=False)
            ctx.digest(proof, out=dg)
            ctx.verify_fs_batch(proof, result=result, want_chal=False)
            ctx.pack_verdicts(result, out=bitmap)
            p2 = proof.clone()
            ctx.prove_fs_digest_batch(w, r, p2, status.clone(), dg2)
            ctx.verify_fs_bitmap_batch(proof, result.clone(), bm2)
        torch.cuda.synchronize()
        assert torch.equal(p2, proof) and int(dg.item()) == int(dg2.item()) and torch.equal(bitmap, bm2), (n, algo)
        done = float((status == 0).float().mean())
        say(f"[{algo}] n = {n} ({100 * done:.1f} % of the proofs complete)")

        def prove():
            ctx.prove_fs_batch(w, r, proof=proof, status=status, want_chal=False)

        def prove_digest():
            prove()
            ctx.digest(proof, out=dg)

        t = rounds([prove, prove_digest, lambda: ctx.prove_fs_digest_batch(w, r, proof, status, dg)], reps)
        say(f"  prover   alone {t[0]:9.1f} us   + pbh_digest_dev {t[1]:9.1f} us   fused {t[2]:9.1f} us   "
            f"fused - alone {t[2] - t[0]:+7.1f} us   fused / unfused {t[2] / t[1]:.3f}")

        def verify():
            ctx.verify_fs_batch(proof, result=result, want_chal=False)

        def verify_pack():
            verify()
            ctx.pack_verdicts(result, out=bitmap)

        t = rounds([verify, verify_pack, lambda: ctx.verify_fs_bitmap_batch(proof, result, bitmap)], reps)
        say(f"  verifier alone {t[0]:9.1f} us   + pbh_pack_verdicts_dev {t[1]:6.1f} us   fused {t[2]:9.1f} us   "
            f"fused - alone {t[2] - t[0]:+7.1f} us   fused / unfused {t[2] / t[1]:.3f}")
    del w, r, proof, status, result, bitmap, bm2, p2
    torch.cuda.empty_cache()
ctx.set_algo("table")
ctx.close()

say("2. pbh_multi_prove_verify_fs_sharded, PBH_ALGO_TABLE, D_fullpath, 2^24 items per device, median of 7 after 2 warm-up passes")
per = 1 << 24
n_all = torch.cuda.device_count()
for n_dev in sorted({1, n_all}):
    with P.MultiContext(n_dev) as mc:
        for _ in range(2):
            mc.prove_verify_fs_sharded(per * n_dev)
        ms = [mc.prove_verify_fs_sharded(per * n_dev)["ms"] for _ in range(7)]
        t = statistics.median(ms)
        say(f"  {n_dev} device(s): {per * n_dev} pairs in {t:8.3f} ms (min {min(ms):.3f}, max {max(ms):.3f})   "
            f"{per * n_dev / t / 1e6:6.3f} G pairs/s, {per / t / 1e6:6.3f} G pairs/s per device")
if n_all == 1:
    say("  more than one device: not measured (one visible device)")

os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "w") as f:
    f.write("\n".join(lines) + "\n")
