"""Host transport of the asynchronous lane calls (include/pbh_b200.h "lanes"): the byte-plane, packed and Fiat-Shamir packed
families enqueued on the same lanes with no synchronisation between calls.  They share one lane buffer per lane, whose rows
each family lays out in its own way and which grows as larger layouts arrive, and the packed verifier may read the proofs the
packed prover left there (PBH_OPT_PROOF_RESIDENT).  Every output byte is compared with the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N = 30011   # ragged: not a multiple of the 256-item tile nor of 16
LANES = 2
_EXPECT = {}


def _words(pk):
    return np.stack([pk["points_lo"], pk["points_hi"], pk["evals_status"]], axis=1)


def _expect(oracle, lane):
    """Inputs and oracle outputs of one lane: byte planes, packed records and Fiat-Shamir packed records, three seeds."""
    import pbh_b200 as P
    if lane not in _EXPECT:
        gen = lambda seed: oracle.generate_inputs(N, first_index=lane * N, seed=seed, dist=1, threads=8)[:4]
        w, r, c, u = gen(70 + lane)
        po, so = oracle.prove_batch(w, r, c, threads=8)
        vo, go = oracle.verify_batch(po, c, u, threads=8)
        planes = dict(w=w, r=r, c=c, u=u, proof=po, status=so, result=vo, gt=go)
        w, r, c, u = gen(80 + lane)
        po, so = oracle.prove_batch(w, r, c, threads=8)
        vo, _ = oracle.verify_batch(po, c, u, threads=8)
        packed = dict(pin=P.pack_witness(w, r, c, u), cu=P.pack_chal_u(c, u), out=oracle.packed_pack_proofs(po, so), res=vo)
        w, r, _, _ = gen(90 + lane)
        po, so, co = oracle.prove_fs_batch(w, r, threads=8)
        vo, _ = oracle.verify_fs_batch(po, threads=8)
        fs = dict(pin=P.pack_fs_witness(w, r), out=oracle.packed_pack_proofs(po, so), cu=oracle.packed_pack_chal_u(co[:5], co[5]), res=vo)
        _EXPECT[lane] = (planes, packed, fs)
    return _EXPECT[lane]


@pytest.mark.parametrize("resident", [1, 0])
def test_families_mixed_on_lanes(oracle, product_lib, resident):
    """On two lanes, in this order and with no synchronisation: byte-plane prove; packed prove; Fiat-Shamir packed prove; packed
    verify of the packed prove's output (not resident: a call came in between); packed prove and at once packed verify of its
    output (resident when the option is on); Fiat-Shamir packed verify; byte-plane verify of the byte-plane proofs.  A fresh
    context, so every lane buffer starts empty and grows from family to family."""
    import pbh_b200 as P
    with P.Context(device=0) as ctx:
        ctx.set_option(P.OPT_PROOF_RESIDENT, resident)
        bufs = []
        for lane in range(LANES):
            planes, packed, fs = _expect(oracle, lane)
            b = dict(w=ctx.host_alloc((12, N)), r=ctx.host_alloc((9, N)), c=ctx.host_alloc((5, N)), u=ctx.host_alloc((N,)),
                     proof=ctx.host_alloc((27, N)), status=ctx.host_alloc((N,)), result=ctx.host_alloc((N,)), gt=ctx.host_alloc((4, N)),
                     pin=ctx.host_alloc_as(N, P.PACKED_WITNESS), cu=ctx.host_alloc_as(N, "<u4"),
                     out=ctx.host_alloc_as(N, P.PACKED_PROOF), res=ctx.host_alloc_as(N, np.uint8),
                     out2=ctx.host_alloc_as(N, P.PACKED_PROOF), res2=ctx.host_alloc_as(N, np.uint8),
                     fs_pin=ctx.host_alloc_as(N, P.PACKED_FS_WITNESS), fs_out=ctx.host_alloc_as(N, P.PACKED_PROOF),
                     fs_cu=ctx.host_alloc_as(N, "<u4"), fs_res=ctx.host_alloc_as(N, np.uint8))
            for k in ("w", "r", "c", "u"):
                b[k][...] = planes[k]
            b["pin"][...] = packed["pin"]; b["cu"][...] = packed["cu"]; b["fs_pin"][...] = fs["pin"]
            for k in ("proof", "status", "result", "gt", "res", "res2", "fs_res"):
                b[k].view(np.uint8)[...] = 0xEE
            for k in ("out", "out2", "fs_out", "fs_cu"):
                b[k].view(np.uint8)[...] = 0xEE
            bufs.append(b)
        steps = [
            lambda l, b: ctx.prove_batch_async(l, b["w"], b["r"], b["c"], b["proof"], b["status"]),
            lambda l, b: ctx.prove_packed_async(l, b["pin"], b["out"]),
            lambda l, b: ctx.prove_fs_packed_async(l, b["fs_pin"], b["fs_out"], b["fs_cu"]),
            lambda l, b: ctx.verify_packed_async(l, b["out"], b["cu"], b["res"]),
            lambda l, b: (ctx.prove_packed_async(l, b["pin"], b["out2"]), ctx.verify_packed_async(l, b["out2"], b["cu"], b["res2"])),
            lambda l, b: ctx.verify_fs_packed_async(l, b["fs_out"], b["fs_res"]),
            lambda l, b: ctx.verify_batch_async(l, b["proof"], b["c"], b["u"], b["result"], gt=b["gt"]),
        ]
        for step in steps:
            for lane in range(LANES):
                step(lane, bufs[lane])
        ctx.sync()
        for lane, b in enumerate(bufs):
            planes, packed, fs = _expect(oracle, lane)
            for k in ("proof", "status", "result", "gt"):
                assert np.array_equal(b[k], planes[k]), (lane, k)
            for k in ("out", "out2"):
                assert np.array_equal(_words(b[k]), packed["out"]), (lane, k)
            assert np.array_equal(b["res"], packed["res"]) and np.array_equal(b["res2"], packed["res"]), lane
            assert np.array_equal(_words(b["fs_out"]), fs["out"]) and np.array_equal(b["fs_cu"], fs["cu"]), lane
            assert np.array_equal(b["fs_res"], fs["res"]), lane
        for b in bufs:
            for arr in b.values():
                ctx.host_free(arr)
