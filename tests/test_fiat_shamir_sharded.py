"""Fiat-Shamir across GPUs (include/pbh_b200.h): the shard summaries fused into the Fiat-Shamir kernels
(pbh_prove_fs_digest_batch_dev, pbh_verify_fs_bitmap_batch_dev), the Fiat-Shamir multi-device calls (pbh_multi_*_fs_*) and the
sharded pass, in Python as sharding.gpu_compute_fs.

Each fused call is defined as the plain Fiat-Shamir call followed by pbh_digest_dev / pbh_pack_verdicts_dev, and is compared with
exactly that, byte for byte; the plain calls are pinned against the oracle by tests/test_fiat_shamir.py, and a strided sample
of a 2^20 batch is compared with the oracle here as well."""
import ctypes as C
import os
import re
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("pbh_prove_fs_digest_batch_dev", "pbh_verify_fs_bitmap_batch_dev", "pbh_multi_prove_fs_batch", "pbh_multi_verify_fs_batch",
       "pbh_multi_prove_fs_packed", "pbh_multi_verify_fs_packed", "pbh_multi_prove_verify_fs_sharded")
M64 = 2**64 - 1


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_new_entry_points_are_declared_bound_and_listed():
    import pbh_b200
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "pbh_b200.h")).read(), flags=re.S)
    ffi = open(os.path.join(ROOT, "plonk-by-fingers_b200", "rust", "src", "ffi.rs")).read()
    for name in NEW:
        assert re.search(r"\bint %s\s*\(" % name, hdr), name
        assert re.search(r"pub fn %s\s*\(" % name, ffi), name
        assert name in pbh_b200.EXPORTS, name
    assert re.search(r"#define PBH_ABI_VERSION 4\b", hdr)


def _oracle_fs_compute(first, count):
    """The Fiat-Shamir shard of sharding.gpu_compute_fs, restated with the oracle."""
    import torch
    import oracle as O
    w, r, _, _, _ = O.generate_inputs(count, first_index=first, seed=0xB200, dist=1)
    proof, _, _ = O.prove_fs_batch(w, r)
    res, _ = O.verify_fs_batch(proof)
    d = O.digest(proof, first_index=first)
    d = d - 2**64 if d >= 2**63 else d
    return torch.from_numpy(O.pack_verdicts(res)), torch.tensor([d], dtype=torch.int64)


def _gloo_worker(rank, world, port, n_total, out_dir):
    sys.path[:0] = [os.path.join(ROOT, "plonk-by-fingers_b200", "python"), os.path.join(ROOT, "oracle")]
    import torch
    import torch.distributed as dist
    from pbh_b200 import sharding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    bitmap, digs, total = sharding.run_sharded(n_total, rank, world, _oracle_fs_compute)
    torch.save({"bitmap": bitmap, "digs": digs, "total": total}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_fs_gather_is_shard_count_independent(tmp_path, oracle):
    """run_sharded over gloo with world sizes 1, 2 and 3 and an oracle-backed Fiat-Shamir shard: every rank of every world size
    ends up with the same bitmap and total digest, and those are the whole batch's."""
    import torch
    import torch.multiprocessing as mp
    from pbh_b200 import sharding
    n_total = 1001
    bitmap1, digs1, total1 = sharding.run_sharded(n_total, 0, 1, _oracle_fs_compute)
    w, r, _, _, _ = oracle.generate_inputs(n_total, first_index=0, seed=0xB200, dist=1)
    proof, _, _ = oracle.prove_fs_batch(w, r)
    res, _ = oracle.verify_fs_batch(proof)
    assert np.array_equal(bitmap1.numpy(), oracle.pack_verdicts(res)) and total1 == oracle.digest(proof) & M64
    for world in (2, 3):
        out = tmp_path / str(world)
        out.mkdir()
        mp.spawn(_gloo_worker, args=(world, _free_port(), n_total, str(out)), nprocs=world, join=True)
        for rank in range(world):
            o = torch.load(os.path.join(out, f"r{rank}.pt"))
            assert torch.equal(o["bitmap"], bitmap1) and o["total"] == total1 and o["digs"].numel() == world, (world, rank)


# ---------------------------------------------------------------------------------------------------------------- GPU
SIZES_PROVE = (1, 31, 32, 33, 255, 70003, (1 << 18) + 4097)
FIRSTS = (0, 2**32 - 5, 2**40 + 3)
SIZES_VERIFY = (1, 7, 8, 9, 31, 32, 33, 70003)


def _inputs(ctx, n, dist, seed, first_index=0):
    """Generated witnesses with zero-blinder rows and out-of-field bytes mixed in, so that every status class occurs."""
    import torch
    w, r, _, _ = ctx.generate_inputs(n, first_index=first_index, seed=seed, dist=dist)
    rng = np.random.default_rng(seed + n + dist)
    m = (n + 9) // 10
    zr = torch.from_numpy(rng.choice(np.array([0, 0, 1, 16, 5], dtype=np.uint8), size=(9, m))).to(r.device)
    r[:, :m] = zr
    bad = rng.random(n) < 0.03
    cols = torch.from_numpy(np.nonzero(bad)[0]).to(w.device)
    if cols.numel():
        w[int(rng.integers(0, 12)), cols] = 17 + int(rng.integers(0, 200))
        r[int(rng.integers(0, 9)), cols[::2]] = 255
    return w, r


def _garbage_digest():
    import torch
    return torch.tensor([0x5A5A5A5A12345678], dtype=torch.int64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ("table", "table_generic", "arith", "table_int"))
def test_fused_digest_equals_prover_plus_digest(gpu_ctx, variant):
    """pbh_prove_fs_digest_batch_dev == pbh_prove_fs_batch_dev + pbh_digest_dev: proof, status and challenge planes byte-equal,
    digest equal and overwritten (the word starts as garbage; no memset in front).  table_int: the int32 prover's fallback."""
    import torch
    ctx = gpu_ctx[variant]
    classes = set()
    for n in SIZES_PROVE:
        for dist in (0, 1):
            w, r = _inputs(ctx, n, dist, seed=7)
            pa = torch.full((27, n), 0xEE, dtype=torch.uint8, device="cuda"); sa = torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")
            ca = torch.full((6, n), 0xEE, dtype=torch.uint8, device="cuda")
            ctx.prove_fs_batch(w, r, proof=pa, status=sa, chal=ca)
            for k, first in enumerate(FIRSTS):
                want = ctx.digest(pa, first_index=first)
                pb = torch.full((27, n), 0xDD, dtype=torch.uint8, device="cuda"); sb = torch.full((n,), 0xDD, dtype=torch.uint8, device="cuda")
                cb = torch.full((6, n), 0xDD, dtype=torch.uint8, device="cuda") if k != 1 else None   # chal_out = NULL: u not derived
                dg = _garbage_digest()
                ctx.prove_fs_digest_batch(w, r, pb, sb, dg, first_index=first, chal=cb)
                ctx.sync()
                assert torch.equal(pb, pa) and torch.equal(sb, sa), (variant, n, dist, first)
                if cb is not None:
                    assert torch.equal(cb, ca), (variant, n, dist, first)
                assert int(dg.item()) == int(want.item()), (variant, n, dist, first)
            classes.update(int(x) for x in torch.unique(sa).tolist())
    assert {0, 32} <= classes and len(classes) >= 4, classes
    dg = _garbage_digest()
    e = torch.empty((12, 0), dtype=torch.uint8, device="cuda")
    ctx.prove_fs_digest_batch(e, torch.empty((9, 0), dtype=torch.uint8, device="cuda"), torch.empty((27, 0), dtype=torch.uint8, device="cuda"),
                              torch.empty((0,), dtype=torch.uint8, device="cuda"), dg)
    ctx.sync()
    assert int(dg.item()) == 0


def _proof_sets(ctx, n):
    """Honest proofs, tampered proofs (evaluations shifted, coordinates out of the field) and all-zero proofs."""
    import torch
    w, r = _inputs(ctx, n, 1, seed=19)
    honest, _ = ctx.prove_fs_batch(w, r, want_chal=False)
    tampered = honest.clone()
    tampered[20 + n % 7, ::3] = (tampered[20 + n % 7, ::3] + 1) % 17
    tampered[2, 1::5] = 200
    tampered[18, 2::7] ^= 0x80
    return {"honest": honest, "tampered": tampered, "zero": torch.zeros((27, n), dtype=torch.uint8, device="cuda")}


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ("table", "arith"))
def test_fused_bitmap_equals_verifier_plus_pack(gpu_ctx, algo):
    """pbh_verify_fs_bitmap_batch_dev == pbh_verify_fs_batch_dev + pbh_pack_verdicts_dev, with the bitmap 4-byte aligned (fused)
    and at an odd address (second kernel), inside a guard-filled buffer whose other bytes stay untouched."""
    import torch
    ctx = gpu_ctx[algo]
    accepted = 0
    for n in SIZES_VERIFY:
        nb = (n + 7) // 8
        for kind, proof in _proof_sets(ctx, n).items():
            want_res = ctx.verify_fs_batch(proof, want_chal=False)
            want_bm = ctx.pack_verdicts(want_res)
            for off in (0, 1):
                buf = torch.full((nb + 16,), 0xA5, dtype=torch.uint8, device="cuda")
                res = torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")
                ctx.verify_fs_bitmap_batch(proof, res, buf[off:off + nb])
                ctx.sync()
                assert torch.equal(res, want_res), (algo, n, kind, off)
                assert torch.equal(buf[off:off + nb], want_bm), (algo, n, kind, off)
                assert bool((buf[:off] == 0xA5).all()) and bool((buf[off + nb:] == 0xA5).all()), (algo, n, kind, off)
            accepted += int((want_res == 1).sum().item())
    # set bits were compared too: how many proofs of a small batch the Fiat-Shamir transcript accepts is the oracle's business,
    # so only the whole run is asked to contain some
    assert accepted > 0, algo


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ("table", "arith"))
def test_fused_calls_equal_the_oracle(gpu_ctx, oracle, algo):
    """A 2^20 D_fullpath batch through the fused calls; a strided sample of 2^16 items against the oracle's Fiat-Shamir prover
    and verifier (status, proof bytes, verdict bit), and the launch's digest against the oracle's digest of the proof bytes."""
    import torch
    ctx = gpu_ctx[algo]
    n, first = 1 << 20, 3 * 2**32 + 17
    w, r = _inputs(ctx, n, 1, seed=5, first_index=first)
    proof = torch.empty((27, n), dtype=torch.uint8, device="cuda"); status = torch.empty((n,), dtype=torch.uint8, device="cuda")
    result = torch.empty((n,), dtype=torch.uint8, device="cuda"); bitmap = torch.empty((n // 8,), dtype=torch.uint8, device="cuda")
    dg = _garbage_digest()
    ctx.prove_fs_digest_batch(w, r, proof, status, dg, first_index=first)
    ctx.verify_fs_bitmap_batch(proof, result, bitmap)
    ctx.sync()
    idx = np.arange(0, n, 16)
    wo, ro = w.cpu().numpy()[:, idx].copy(), r.cpu().numpy()[:, idx].copy()
    threads = max(1, oracle.hardware_threads())
    po, so, _ = oracle.prove_fs_batch(wo, ro, threads=threads)
    vo, _ = oracle.verify_fs_batch(po, threads=threads)
    hp = proof.cpu().numpy()
    assert np.array_equal(status.cpu().numpy()[idx], so) and np.array_equal(hp[:, idx], po)
    bits = np.unpackbits(bitmap.cpu().numpy(), bitorder="little")
    assert np.array_equal(bits[idx], vo & 1) and np.array_equal(result.cpu().numpy()[idx], vo)
    assert int(dg.item()) & M64 == oracle.digest(hp, first_index=first) & M64
    # per item: the sample's digests, restated by the oracle from its own proofs, sum to the digest of the GPU's sampled columns
    per_item = sum(oracle.digest(po[:, k:k + 1], first_index=first + int(i)) for k, i in enumerate(idx[:4096])) & M64
    assert per_item == sum(oracle.digest(hp[:, i:i + 1], first_index=first + int(i)) for i in idx[:4096]) & M64


@pytest.mark.gpu
def test_shard_count_independence_on_one_gpu(gpu_ctx):
    """One 2^20 + 13 batch cut into 1, 2, 3 and 7 shards at multiples of 8 items, each shard with its own first_index: the
    concatenated bitmaps and the summed digests equal the whole-batch call."""
    import torch
    from pbh_b200 import sharding
    ctx = gpu_ctx["table"]
    n, first = (1 << 20) + 13, 1000 * 8
    w, r = _inputs(ctx, n, 1, seed=23, first_index=first)

    def run(lo, hi):
        m = hi - lo
        proof = torch.empty((27, m), dtype=torch.uint8, device="cuda"); status = torch.empty((m,), dtype=torch.uint8, device="cuda")
        result = torch.empty((m,), dtype=torch.uint8, device="cuda")
        bitmap = torch.empty(((m + 7) // 8,), dtype=torch.uint8, device="cuda"); dg = _garbage_digest()
        ctx.prove_fs_digest_batch(w[:, lo:hi], r[:, lo:hi], proof, status, dg, first_index=first + lo)
        ctx.verify_fs_bitmap_batch(proof, result, bitmap)
        return bitmap, dg

    whole_bm, whole_dg = run(0, n)
    ctx.sync()
    for shards in (1, 2, 3, 7):
        parts = [run(*sharding.shard_range(n, k, shards)) for k in range(shards)]
        ctx.sync()
        assert torch.equal(torch.cat([b for b, _ in parts]), whole_bm), shards
        assert sum(int(d.item()) & M64 for _, d in parts) & M64 == int(whole_dg.item()) & M64, shards


@pytest.mark.gpu
def test_fused_calls_replay_from_a_cuda_graph(gpu_ctx):
    """The fused prover and verifier captured once and replayed twice on each of two streams: every replay overwrites the
    digest and the bitmap with the direct call's values (the launch-local record is re-armed by the last block)."""
    import torch
    for algo in ("table", "arith"):
        ctx = gpu_ctx[algo]
        n = (1 << 18) + 77
        w, r = _inputs(ctx, n, 1, seed=41)
        proof = torch.empty((27, n), dtype=torch.uint8, device="cuda"); status = torch.empty((n,), dtype=torch.uint8, device="cuda")
        result = torch.empty((n,), dtype=torch.uint8, device="cuda"); bitmap = torch.empty(((n + 7) // 8,), dtype=torch.uint8, device="cuda")
        dg = _garbage_digest()
        ctx.prove_fs_digest_batch(w, r, proof, status, dg, first_index=99)
        ctx.verify_fs_bitmap_batch(proof, result, bitmap)
        ctx.sync()
        want_dg, want_bm = int(dg.item()), bitmap.clone()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=torch.cuda.Stream()):
            ctx.prove_fs_digest_batch(w, r, proof, status, dg, first_index=99)
            ctx.verify_fs_bitmap_batch(proof, result, bitmap)
        torch.cuda.synchronize()
        for st in (torch.cuda.Stream(), torch.cuda.Stream()):
            with torch.cuda.stream(st):
                dg.fill_(0x1234567)
                bitmap.fill_(0xA5)
                for _ in range(2):
                    g.replay()
            st.synchronize()
            assert int(dg.item()) == want_dg and torch.equal(bitmap, want_bm), algo
        del g


@pytest.mark.gpu
def test_peer_window_replicates_the_fs_summaries(gpu_ctx):
    """Two ranks of one process on cuda:0 (pbh_window_attach_ptrs): the digest and bitmap the Fiat-Shamir calls write into the
    own row appear at the same offset of the peer's window - fused (FP32 prover, aligned bitmap) and through the fallbacks (int32
    prover, bitmap at an odd address) - and equal digest / pack_verdicts.  A summary outside the own row is not replicated."""
    import torch
    import pbh_b200
    world, n = 2, 256 * 37 + 64 + 5
    nb = (n + 7) // 8
    dofs = (nb + 1 + 7) // 8 * 8            # digest offset in a slot, after a bitmap that may start at byte 1
    slot = (dofs + 8 + 15) // 16 * 16
    ranks = [pbh_b200.Context(device=0, algo="table") for _ in range(world)]
    try:
        wins = [c.window_create(3 * slot, k, world)[0] for k, c in enumerate(ranks)]
        for c in ranks:
            c.window_attach_ptrs([c2._window_base for c2 in ranks])
        ref = gpu_ctx["table"]
        for k, c in enumerate(ranks):
            first = k * n
            w, r = _inputs(ref, n, 1, seed=57 + k, first_index=first)
            ref.sync()
            proof = torch.empty((27, n), dtype=torch.uint8, device="cuda"); status = torch.empty((n,), dtype=torch.uint8, device="cuda")
            result = torch.empty((n,), dtype=torch.uint8, device="cuda")
            for s, (fp32, off) in enumerate(((1, 0), (0, 1))):
                c.set_option(pbh_b200.OPT_PROVER_FP32, fp32)
                mine = wins[k][k, s * slot:(s + 1) * slot]
                c.prove_fs_digest_batch(w, r, proof, status, mine[dofs:dofs + 8].view(torch.int64), first_index=first)
                c.verify_fs_bitmap_batch(proof, result, mine[off:off + nb])
                c.sync()
                want_bm = ref.pack_verdicts(result); want_dg = ref.digest(proof, first_index=first)
                ref.sync()
                for holder in range(world):
                    got = wins[holder][k, s * slot:(s + 1) * slot]
                    assert torch.equal(got[off:off + nb], want_bm), (k, s, holder)
                    assert int(got[dofs:dofs + 8].view(torch.int64).item()) == int(want_dg.item()), (k, s, holder)
            c.set_option(pbh_b200.OPT_PROVER_FP32, 1)
            other = wins[k][1 - k, 2 * slot:3 * slot]
            before = wins[1 - k][1 - k, 2 * slot:3 * slot].clone()
            c.prove_fs_digest_batch(w, r, proof, status, other[dofs:dofs + 8].view(torch.int64), first_index=first)
            c.verify_fs_bitmap_batch(proof, result, other[:nb])
            c.sync()
            assert torch.equal(other[:nb], want_bm) and int(other[dofs:dofs + 8].view(torch.int64).item()) == int(want_dg.item())
            assert torch.equal(wins[1 - k][1 - k, 2 * slot:3 * slot], before)
    finally:
        for c in ranks:
            c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ("table", "arith"))
def test_multi_device_fs_calls(gpu_ctx, algo):
    """pbh_multi_*_fs_* on every visible GPU (one on a single-GPU box): the host-pointer plane and packed calls equal the
    single-context calls; the sharded pass equals one context computing the same global range with the fused `_dev` calls."""
    import torch
    import pbh_b200
    n_dev = min(torch.cuda.device_count(), 8)
    ctx = gpu_ctx[algo]
    with pbh_b200.MultiContext(n_dev, algo=algo) as mc:
        n = 3 * 256 * n_dev + 77
        wd, rd = _inputs(ctx, n, 0, seed=61)
        w, r = wd.cpu().numpy(), rd.cpu().numpy()
        p, s, ch = mc.prove_fs_batch(w, r)
        p1, s1, ch1 = ctx.prove_fs_batch(w, r)
        assert np.array_equal(p, p1) and np.array_equal(s, s1) and np.array_equal(ch, ch1)
        v, cv, g = mc.verify_fs_batch(p, want_chal=True, want_gt=True)
        v1, cv1, g1 = ctx.verify_fs_batch(p, want_chal=True, want_gt=True)
        assert np.array_equal(v, v1) and np.array_equal(cv, cv1) and np.array_equal(g, g1)
        assert np.array_equal(mc.verify_fs_batch(p), v1)
        pin = pbh_b200.pack_fs_witness(w % 17, r % 17)
        pk, cu = mc.prove_fs_packed(pin)
        pk1, cu1 = ctx.prove_fs_packed(pin)
        assert np.array_equal(pk, pk1) and np.array_equal(cu, cu1)
        assert np.array_equal(mc.verify_fs_packed(pk), ctx.verify_fs_packed(pk))
        for n_total, first in ((3 * 256 * n_dev + 77, 0), ((1 << 20) + 5, 12345 * 8)):
            out = mc.prove_verify_fs_sharded(n_total, first_index=first, seed=0xB200)
            gw, gr, _, _ = ctx.generate_inputs(n_total, first_index=first, seed=0xB200, dist=1)
            proof = torch.empty((27, n_total), dtype=torch.uint8, device="cuda"); status = torch.empty((n_total,), dtype=torch.uint8, device="cuda")
            result = torch.empty((n_total,), dtype=torch.uint8, device="cuda")
            bitmap = torch.empty(((n_total + 7) // 8,), dtype=torch.uint8, device="cuda"); dg = _garbage_digest()
            ctx.prove_fs_digest_batch(gw, gr, proof, status, dg, first_index=first)
            ctx.verify_fs_bitmap_batch(proof, result, bitmap)
            ctx.sync()
            bm = bitmap.cpu().numpy()
            assert np.array_equal(out["bitmap"], bm), (algo, n_total)
            assert out["total_digest"] == int(dg.item()) & M64 and sum(int(x) for x in out["digests"]) & M64 == out["total_digest"]
            assert out["accepted"] == int(np.unpackbits(bm).sum()) == int((result == 1).sum().item()) and out["ms"] > 0


def _nccl_fs_worker(rank, world, port, n_total, out_dir):
    sys.path[:0] = [os.path.join(ROOT, "plonk-by-fingers_b200", "python")]
    import torch
    import torch.distributed as dist
    import pbh_b200
    from pbh_b200 import sharding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ctx = pbh_b200.Context(device=rank)
    bitmap, digs, total = sharding.run_sharded(n_total, rank, world, lambda lo, cnt: sharding.gpu_compute_fs(ctx, lo, cnt))
    torch.save({"bitmap": bitmap.cpu(), "digs": digs.cpu(), "total": total}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.barrier()
    torch.cuda.synchronize()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_run_sharded_fs_under_real_nccl(gpu_ctx, tmp_path):
    """run_sharded with gpu_compute_fs, one process per GPU over NCCL: every rank's bitmap and total digest equal one GPU's."""
    import torch
    import torch.multiprocessing as mp
    from pbh_b200 import sharding
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip(f"needs >= 2 visible GPUs for NCCL ranks, this box shows {torch.cuda.device_count()} "
                    "(shard-count independence on one GPU: test_shard_count_independence_on_one_gpu)")
    n_total = (1 << 20) + 4000 + 5
    sb, _, st = sharding.run_sharded(n_total, 0, 1, lambda lo, cnt: sharding.gpu_compute_fs(gpu_ctx["table"], lo, cnt))
    mp.spawn(_nccl_fs_worker, args=(world, _free_port(), n_total, str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        o = torch.load(os.path.join(tmp_path, f"r{rank}.pt"))
        assert torch.equal(o["bitmap"], sb.cpu()) and o["total"] == st and o["digs"].numel() == world


@pytest.mark.gpu
def test_argument_errors(gpu_ctx, product_lib):
    import torch
    import pbh_b200
    lib, ctx = product_lib, gpu_ctx["table"]
    n = 64
    buf = torch.zeros((64, n), dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    dg = torch.zeros((1,), dtype=torch.int64, device="cuda")
    sz = C.c_size_t

    def prove(wit=p(buf), wp=n, rnd=p(buf[12]), rp=n, proof=p(buf[21]), pp=n, status=p(buf[48]), chal=None, cp=0, digest=p(dg), count=n, h=ctx.h):
        return lib.pbh_prove_fs_digest_batch_dev(h, sz(count), wit, sz(wp), rnd, sz(rp), proof, sz(pp), status, chal, sz(cp),
                                                 C.c_uint64(0), digest)

    def verify(proof=p(buf), pp=n, result=p(buf[30]), bitmap=p(buf[31]), count=n, h=ctx.h):
        return lib.pbh_verify_fs_bitmap_batch_dev(h, sz(count), proof, sz(pp), result, bitmap)

    assert prove() == 0 and verify() == 0
    ctx.sync()
    for kw in (dict(wit=None), dict(rnd=None), dict(proof=None), dict(status=None), dict(digest=None), dict(digest=None, count=0),
               dict(wp=n - 1), dict(rp=n - 1), dict(pp=n - 1), dict(chal=p(buf[50]), cp=n - 1), dict(h=None)):
        assert prove(**kw) == -1, kw
    for kw in (dict(proof=None), dict(result=None), dict(bitmap=None), dict(pp=n - 1), dict(h=None)):
        assert verify(**kw) == -1, kw
    with pbh_b200.MultiContext(1) as mc:
        m, nul = mc.h, None
        assert lib.pbh_multi_prove_fs_batch(m, sz(n), nul, sz(n), p(buf), sz(n), p(buf), sz(n), p(buf), nul, sz(0)) == -1
        assert lib.pbh_multi_verify_fs_batch(m, sz(n), nul, sz(n), p(buf), nul, sz(0), nul, sz(0)) == -1
        assert lib.pbh_multi_prove_fs_packed(m, sz(n), nul, nul, nul) == -1
        assert lib.pbh_multi_verify_fs_packed(m, sz(n), nul, nul) == -1
        assert lib.pbh_multi_prove_verify_fs_sharded(m, C.c_uint64(n), C.c_uint64(0), C.c_uint64(0), 1, nul, nul, nul, nul, nul) == -1
        with pytest.raises(pbh_b200.PbhError):
            mc.prove_fs_batch(np.zeros((12, n), np.uint8), np.zeros((8, n), np.uint8))
