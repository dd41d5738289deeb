"""Sharding of a proof batch over ranks (one process per GPU) — SURVEY.md §8e.

Proofs are independent, so the batch partitions into contiguous index ranges with no data-path collective.  The
only exchange is at the end: an all-gather of each shard's verdict bitmap (1 bit per proof) and of its additive
64-bit proof digest.  Results are identical for every shard count: item bytes depend only on (seed, global index),
bitmaps concatenate (shard boundaries are multiples of 8 items) and digests add modulo 2^64.

`compute(first_index, count)` does the per-shard work and returns (bitmap uint8 tensor of ceil(count/8) bytes,
digest int64 tensor of 1 element).  On a GPU rank it is `gpu_compute(ctx, ...)` below, or `gpu_compute_fs(ctx, ...)` for
the Fiat-Shamir transcript (CUDA kernels through the C ABI); the CPU tests pass an oracle-backed stand-in to exercise this host logic under gloo.
"""
import torch


def shard_range(n_total, rank, world):
    """Contiguous range [lo, hi) of `rank`; every boundary except the last is a multiple of 8 items."""
    per = -(-n_total // world)
    per = -(-per // 8) * 8
    lo = min(n_total, rank * per)
    hi = min(n_total, lo + per)
    return lo, hi


def shard_bytes(n_total, world):
    per = -(-n_total // world)
    per = -(-per // 8) * 8
    return per // 8


def gather_summaries(bitmap, digest, n_total, world, group=None):
    """All-gather shard bitmaps and digests; returns (global bitmap uint8[ceil(n/8)], per-shard digests int64[world],
    total digest as a Python int modulo 2^64)."""
    nb = shard_bytes(n_total, world)
    padded = torch.zeros(nb, dtype=torch.uint8, device=bitmap.device)
    padded[: bitmap.numel()] = bitmap
    if world == 1:
        bits, digs = padded.unsqueeze(0), digest.reshape(1, 1)
    else:
        import torch.distributed as dist
        flat_bits = torch.empty(world * nb, dtype=torch.uint8, device=bitmap.device)   # flat: gloo and nccl both accept it
        flat_digs = torch.empty(world, dtype=torch.int64, device=bitmap.device)
        dist.all_gather_into_tensor(flat_bits, padded, group=group)
        dist.all_gather_into_tensor(flat_digs, digest.reshape(1), group=group)
        bits, digs = flat_bits.view(world, nb), flat_digs.view(world, 1)
    parts = []
    for r in range(world):
        lo, hi = shard_range(n_total, r, world)
        parts.append(bits[r, : (hi - lo + 7) // 8])
    total = sum(int(d) & (2**64 - 1) for d in digs.reshape(-1).tolist()) % 2**64
    return torch.cat(parts), digs.reshape(-1), total


def gpu_compute(ctx, first_index, count, seed=0xB200, dist_kind=1):
    """One shard on this rank's GPU: generate -> prove -> verify -> pack verdicts -> digest proofs (all CUDA)."""
    w, r, c, u = ctx.generate_inputs(count, first_index=first_index, seed=seed, dist=dist_kind)
    import torch
    dev = w.device
    proof = torch.empty((27, count), dtype=torch.uint8, device=dev); status = torch.empty((count,), dtype=torch.uint8, device=dev)
    result = torch.empty((count,), dtype=torch.uint8, device=dev)
    bitmap = torch.empty(((count + 7) // 8 + 3) // 4 * 4, dtype=torch.uint8, device=dev)[: (count + 7) // 8]
    digest = torch.empty((1,), dtype=torch.int64, device=dev)
    ctx.prove_digest_batch(w, r, c, proof, status, digest, first_index=first_index)   # digest fused into the prover
    ctx.verify_bitmap_batch(proof, c, u, result, bitmap)                              # bitmap fused into the verifier
    ctx.sync()
    return bitmap, digest


def gpu_compute_fs(ctx, first_index, count, seed=0xB200, dist_kind=1):
    """gpu_compute with the Fiat-Shamir transcript: the challenges and u are derived from the proofs, so the generated ones
    are not used."""
    w, r, _, _ = ctx.generate_inputs(count, first_index=first_index, seed=seed, dist=dist_kind)
    import torch
    dev = w.device
    proof = torch.empty((27, count), dtype=torch.uint8, device=dev); status = torch.empty((count,), dtype=torch.uint8, device=dev)
    result = torch.empty((count,), dtype=torch.uint8, device=dev)
    bitmap = torch.empty(((count + 7) // 8 + 3) // 4 * 4, dtype=torch.uint8, device=dev)[: (count + 7) // 8]
    digest = torch.empty((1,), dtype=torch.int64, device=dev)
    ctx.prove_fs_digest_batch(w, r, proof, status, digest, first_index=first_index)
    ctx.verify_fs_bitmap_batch(proof, result, bitmap)
    ctx.sync()
    return bitmap, digest


def run_sharded(n_total, rank, world, compute, group=None):
    lo, hi = shard_range(n_total, rank, world)
    bitmap, digest = compute(lo, hi - lo)
    return gather_summaries(bitmap, digest, n_total, world, group)
