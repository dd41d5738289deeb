"""Fiat-Shamir prove / verify over packed records (include/pbh_b200.h "Fiat-Shamir over packed records").

The format is words 0..2 of the packed witness and the packed proof, both pinned by tests/test_packed_format.py against the
oracle's restatement (oracle/oracle.py packed_*).  The content is pinned by definition: pbh_prove_fs_packed(in) =
pack(pbh_prove_fs_batch(unpack(in))) with chal_u_out = pack_chal_u(chal_out), and pbh_verify_fs_packed(p) =
pbh_verify_fs_batch(unpack(p)), both against the oracle's Fiat-Shamir prover and verifier (tests/test_fiat_shamir.py)."""
import ctypes as C

import numpy as np
import pytest

SIZES = (1, 255, 70003, (1 << 18) + 4097)
_EXPECT = {}


def _words(pk):
    return np.stack([pk["points_lo"], pk["points_hi"], pk["evals_status"]], axis=1)


def _inputs(oracle, n, dist, seed=31):
    """Seeded witnesses with zero-blinder rows mixed in (they take the prover's exact-length integer routine)."""
    w, r, _, _, _ = oracle.generate_inputs(n, seed=seed + n, dist=dist, threads=8)
    m = (n + 9) // 10
    r[:, :m] = np.random.default_rng(n + dist).choice(np.array([0, 0, 1, 16, 5], dtype=np.uint8), size=(9, m))
    return w, r


def _expect(oracle, n, dist):
    """(w, r, packed proofs, packed challenge words, verdicts, proof planes) from the oracle, cached across contexts."""
    if (n, dist) not in _EXPECT:
        w, r = _inputs(oracle, n, dist)
        po, so, co = oracle.prove_fs_batch(w, r, threads=8)
        vo, _ = oracle.verify_fs_batch(po, threads=8)
        _EXPECT[(n, dist)] = (w, r, oracle.packed_pack_proofs(po, so), oracle.packed_pack_chal_u(co[:5], co[5]), vo, so)
    return _EXPECT[(n, dist)]


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_fs_witness_host_codec_equals_the_restatement(product_lib, oracle):
    import pbh_b200 as P
    n = 3000
    w, r, _, _, _ = oracle.generate_inputs(n, seed=12, dist=0, threads=4)
    pk = P.pack_fs_witness(w, r)
    assert pk.dtype.itemsize == 12
    want = oracle.packed_pack_witness(w, r, np.zeros((5, n), np.uint8), np.zeros(n, np.uint8))[:, :3]
    assert np.array_equal(pk["w"], want)
    # the same three words as the full packed witness, whatever its challenges
    _, _, c, u, _ = oracle.generate_inputs(n, seed=12, dist=0, threads=4)
    assert np.array_equal(P.pack_witness(w, r, c, u)["w"][:, :3], pk["w"])
    back_w, back_r = P.unpack_fs_witness(pk)
    assert np.array_equal(back_w, w) and np.array_equal(back_r, r)
    # a value >= 17 has no packed form, in either plane
    for planes, k in ((0, 4), (1, 8)):
        bad = [w.copy(), r.copy()]
        bad[planes][k, 5] = 17 + k
        with pytest.raises(P.PbhError):
            P.pack_fs_witness(*bad)
    # arbitrary 32-bit words, >= 17^7 among them, decode as the full witness decodes them with a zero fourth word
    rng = np.random.default_rng(2027)
    rw = rng.integers(0, 2**32, (700, 3), dtype=np.uint64).astype("<u4")
    rw[:5] = [[0, 0, 0], [0xFFFFFFFF] * 3, [17**7 - 1] * 3, [17**7] * 3, [17**7 + 12345, 10 * 17**7, 177 * 17**6]]
    got_w, got_r = P.unpack_fs_witness(rw.view(P.PACKED_FS_WITNESS).reshape(-1))
    ow, orr, _, _ = oracle.packed_unpack_witness(np.concatenate([rw, np.zeros((700, 1), "<u4")], axis=1))
    assert np.array_equal(got_w, ow) and np.array_equal(got_r, orr)
    assert got_w[6, 3] == 17 and got_w[6, 1] >= 17


def test_fs_witness_host_codec_arguments(product_lib):
    lib = product_lib
    buf = np.zeros(64, np.uint8)
    assert lib.pbh_pack_fs_witness_host(C.c_size_t(0), None, C.c_size_t(0), None, C.c_size_t(0), None) == 0
    assert lib.pbh_pack_fs_witness_host(C.c_size_t(1), C.c_void_p(buf.ctypes.data), C.c_size_t(1), None, C.c_size_t(1),
                                        C.c_void_p(buf.ctypes.data)) == -1
    assert lib.pbh_pack_fs_witness_host(C.c_size_t(4), C.c_void_p(buf.ctypes.data), C.c_size_t(3), C.c_void_p(buf.ctypes.data),
                                        C.c_size_t(4), C.c_void_p(buf.ctypes.data)) == -1                    # pitch < n
    assert lib.pbh_unpack_fs_witness_host(C.c_size_t(1), None, None, C.c_size_t(0), None, C.c_size_t(0)) == -1
    # null planes are skipped
    assert lib.pbh_unpack_fs_witness_host(C.c_size_t(1), C.c_void_p(buf.ctypes.data), None, C.c_size_t(0), None, C.c_size_t(0)) == 0


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["table", "arith"])
def test_fs_packed_equals_the_oracle(gpu_ctx, oracle, algo):
    """Device and host calls, both input distributions, ragged sizes and the staged-chunk boundary: the oracle's Fiat-Shamir
    proofs packed, its challenges packed, its verdicts; and the plain packed verifier agrees on every completed proof."""
    import torch
    import pbh_b200 as P
    ctx = gpu_ctx[algo]
    dev = torch.device("cuda", 0)
    seen = set()
    for n in SIZES:
        for dist in (P.DIST_UNIFORM, P.DIST_FULLPATH):
            w, r, want, want_cu, vo, so = _expect(oracle, n, dist)
            pin = P.pack_fs_witness(w, r)
            out_d, cu_d = ctx.prove_fs_packed(torch.from_numpy(pin.view(np.uint8)).to(dev))
            res_d = ctx.verify_fs_packed(out_d)
            ctx.sync()
            out_dn = out_d.cpu().numpy().view(P.PACKED_PROOF)
            assert np.array_equal(_words(out_dn), want), (algo, n, dist)
            assert np.array_equal(cu_d.cpu().numpy().view("<u4"), want_cu), (algo, n, dist)
            assert np.array_equal(res_d.cpu().numpy(), vo), (algo, n, dist)
            out, cu = ctx.prove_fs_packed(pin)
            assert np.array_equal(_words(out), want) and np.array_equal(cu, want_cu), (algo, n, dist)
            assert np.array_equal(ctx.verify_fs_packed(out), vo), (algo, n, dist)
            # without the challenge words (the prover skips the step that derives u): the same proofs
            assert np.array_equal(ctx.prove_fs_packed(pin, want_chal_u=False), out)
            out_d2 = ctx.prove_fs_packed(torch.from_numpy(pin.view(np.uint8)).to(dev), want_chal_u=False)
            ctx.sync()
            assert np.array_equal(out_d2.cpu().numpy().view(P.PACKED_PROOF), out)
            # a completed Fiat-Shamir proof verified with its derived challenges by the plain packed verifier: same verdict
            ok = so == 0
            if ok.any():
                assert np.array_equal(ctx.verify_packed(out[ok], cu[ok]), vo[ok]), (algo, n, dist)
            seen |= set(np.unique(vo).tolist())
    assert {P.VR_ACCEPT, P.VR_REJECT_PAIRING, P.VR_NOT_ON_CURVE}.issubset(seen), seen


@pytest.mark.gpu
def test_fs_packed_prover_variants_and_other_circuit(gpu_ctx, oracle):
    """PBH_OPT_PROVER_FP32 = 0, PBH_OPT_SPECIALISE = 0 and the FP32 verifier give the same bytes; another circuit and SRS give the
    oracle's bytes for that circuit."""
    import pbh_b200 as P
    n = 70003
    w, r, want, want_cu, vo, _ = _expect(oracle, n, P.DIST_UNIFORM)
    pin = P.pack_fs_witness(w, r)
    for name in ("table_int", "arith_int", "table_generic", "table_vf32"):
        out, cu = gpu_ctx[name].prove_fs_packed(pin)
        assert np.array_equal(_words(out), want) and np.array_equal(cu, want_cu), name
        assert np.array_equal(gpu_ctx[name].verify_fs_packed(out), vo), name
    n = 20011
    w, r = _inputs(oracle, n, P.DIST_UNIFORM, seed=5)
    pin = P.pack_fs_witness(w, r)
    ocirc = oracle.pbh_test_circuit(); ocirc.q_c[3] = 2
    pcirc = P.pbh_test_circuit(); pcirc.q_c[3] = 2
    for s, srs_n in ((3, 6), (2, 9)):
        po, so, co = oracle.prove_fs_batch(w, r, circuit=ocirc, s=s, srs_n=srs_n, threads=8)
        vo, _ = oracle.verify_fs_batch(po, circuit=ocirc, s=s, srs_n=srs_n, threads=8)
        for algo in ("table", "arith"):
            with P.Context(circuit=pcirc, s=s, srs_n=srs_n, device=0, algo=algo) as ctx:
                out, cu = ctx.prove_fs_packed(pin)
                assert np.array_equal(_words(out), oracle.packed_pack_proofs(po, so)), (s, srs_n, algo)
                assert np.array_equal(cu, oracle.packed_pack_chal_u(co[:5], co[5])), (s, srs_n, algo)
                assert np.array_equal(ctx.verify_fs_packed(out), vo), (s, srs_n, algo)


@pytest.mark.gpu
def test_fs_packed_verify_of_tampered_words(gpu_ctx, oracle):
    """Words outside the format, tampered digits and every non-zero status code: pbh_verify_fs_packed answers what the oracle's
    Fiat-Shamir verifier answers for the planes the restatement decodes them to."""
    import torch
    import pbh_b200 as P
    rng = np.random.default_rng(19)
    n = 40000
    w, r, _, _, _ = oracle.generate_inputs(n, seed=4, dist=1, threads=8)
    po, so, _ = oracle.prove_fs_batch(w, r, threads=8)
    words = oracle.packed_pack_proofs(po, so).copy()
    k = n // 8
    words[0 * k:1 * k, 0] ^= rng.integers(0, 2**32, k, dtype=np.uint64).astype("<u4")          # other points (still on the curve)
    words[1 * k:2 * k, 1] = rng.integers(0, 2**32, k, dtype=np.uint64).astype("<u4")           # ninth digit mostly >= 102
    words[2 * k:3 * k, 2] = rng.integers(0, 2**29, k, dtype=np.uint64).astype("<u4")           # other evaluations, digits >= 17 among them
    words[3 * k:4 * k, 2] |= ((np.arange(k) % 7) + 1).astype("<u4") << 29                      # every non-zero status code 1..7
    words[4 * k:5 * k] = rng.integers(0, 2**32, (k, 3), dtype=np.uint64).astype("<u4")       # random words
    planes, _ = oracle.packed_unpack_proofs(words)
    want, _ = oracle.verify_fs_batch(planes, threads=8)
    assert len(set(want.tolist())) >= 5
    assert (want[3 * k:4 * k] == P.VR_NOT_ON_CURVE).all()
    recs = words.view(P.PACKED_PROOF).reshape(-1)
    for algo in ("table", "arith", "table_vf32"):
        ctx = gpu_ctx[algo]
        assert np.array_equal(ctx.verify_fs_packed(recs), want), algo
        got = ctx.verify_fs_packed(torch.from_numpy(words.view(np.uint8).reshape(-1)).cuda())
        ctx.sync()
        assert np.array_equal(got.cpu().numpy(), want), algo


@pytest.mark.gpu
def test_fs_packed_prover_words_outside_the_format(gpu_ctx, oracle):
    """A prover word >= 17^7 decodes to a byte >= 17: PBH_ST_BAD_ENCODING, status code 7, zero payload, zero challenge word."""
    import pbh_b200 as P
    rng = np.random.default_rng(23)
    n = 5000
    w, r = _inputs(oracle, n, P.DIST_FULLPATH, seed=8)
    words = P.pack_fs_witness(w, r)["w"].copy()
    bad = np.zeros(n, bool)
    bad[::3] = True
    col = rng.integers(0, 3, n)
    words[bad, col[bad]] = rng.integers(17**7, 2**32, int(bad.sum()), dtype=np.uint64).astype("<u4")
    words[0] = [0xFFFFFFFF, 0, 0]
    words[3] = [0, 0, 17**7]
    ow, orr, _, _ = oracle.packed_unpack_witness(np.concatenate([words, np.zeros((n, 1), "<u4")], axis=1))
    po, so, co = oracle.prove_fs_batch(ow, orr, threads=8)
    assert (so[bad] == P.ST_BAD_ENCODING).all() and (so[~bad] != P.ST_BAD_ENCODING).all()
    recs = words.view(P.PACKED_FS_WITNESS).reshape(-1)
    for algo in ("table", "arith"):
        out, cu = gpu_ctx[algo].prove_fs_packed(recs)
        assert np.array_equal(_words(out), oracle.packed_pack_proofs(po, so)), algo
        assert np.array_equal(cu, oracle.packed_pack_chal_u(co[:5], co[5])), algo
        assert (out["evals_status"][bad] == 7 << 29).all() and not out["points_lo"][bad].any() and not out["points_hi"][bad].any()
        assert not cu[bad].any()


@pytest.mark.gpu
def test_fs_packed_host_paths_and_lanes(gpu_ctx, oracle):
    """Pageable and page-locked memory, small staged chunks, two to four lanes interleaved, the pageable fallback of the lane
    calls: every result equals the device call's."""
    import torch
    import pbh_b200 as P
    ctx = gpu_ctx["table"]
    n = 30011
    sets = []
    for lane in range(4):
        w, r = _inputs(oracle, n, lane % 2, seed=100 + lane)
        pin = P.pack_fs_witness(w, r)
        out_d, cu_d = ctx.prove_fs_packed(torch.from_numpy(pin.view(np.uint8)).cuda())
        res_d = ctx.verify_fs_packed(out_d)
        ctx.sync()
        ref = (out_d.cpu().numpy().view(P.PACKED_PROOF), cu_d.cpu().numpy().view("<u4"), res_d.cpu().numpy())
        b = dict(pin=ctx.host_alloc_as(n, P.PACKED_FS_WITNESS), out=ctx.host_alloc_as(n, P.PACKED_PROOF), cu=ctx.host_alloc_as(n, "<u4"),
                 res=ctx.host_alloc_as(n, np.uint8))
        b["pin"][...] = pin
        sets.append((b, pin, ref))
    # page-locked synchronous calls
    b, pin, (ro, rc, rr) = sets[0]
    ctx.prove_fs_packed(b["pin"], out=b["out"], chal_u=b["cu"])
    ctx.verify_fs_packed(b["out"], result=b["res"])
    assert np.array_equal(b["out"], ro) and np.array_equal(b["cu"], rc) and np.array_equal(b["res"], rr)
    # pageable, in chunks of 256 items (118 chunks over the staging slots)
    with P.Context(device=0) as small:
        small.set_option(P.OPT_CHUNK_LOG2, 8)
        out, cu = small.prove_fs_packed(pin)
        assert np.array_equal(out, ro) and np.array_equal(cu, rc)
        assert np.array_equal(small.verify_fs_packed(out), rr)
        assert np.array_equal(small.prove_fs_packed(pin, want_chal_u=False), ro)
    # lanes: 2, 3 and 4 lanes interleaved, three repetitions each
    for lanes in (2, 3, 4):
        for b, _, _ in sets:
            b["out"].view(np.uint8)[...] = 0xEE; b["cu"][...] = 0xEEEEEEEE; b["res"][...] = 0xEE
        for rep in range(3):
            for lane in range(lanes):
                b = sets[lane][0]
                ctx.lane_sync(lane)
                ctx.prove_fs_packed_async(lane, b["pin"], b["out"], b["cu"] if rep != 1 else None)
                ctx.verify_fs_packed_async(lane, b["out"], b["res"])
        ctx.sync()
        for lane in range(lanes):
            b, _, (ro, rc, rr) = sets[lane]
            assert np.array_equal(b["out"], ro) and np.array_equal(b["cu"], rc) and np.array_equal(b["res"], rr), (lanes, lane)
    # a verify on a lane behind a prove into the same buffer, after the caller changed it: the verifier reads the new contents
    b, _, (ro, _, rr) = sets[1]
    tampered = np.array(ro); tampered[:3000] = tampered[3000:6000]
    want_t = ctx.verify_fs_packed(tampered)
    assert not np.array_equal(want_t, rr)
    b["out"][...] = tampered
    ctx.verify_fs_packed_async(1, b["out"], b["res"])
    ctx.lane_sync(1)
    assert np.array_equal(b["res"], want_t)
    # pageable arrays through the lane entry points: synchronous, same bytes
    _, pin, (ro, rc, rr) = sets[2]
    out = np.zeros(n, P.PACKED_PROOF); cu = np.zeros(n, "<u4"); res = np.zeros(n, np.uint8)
    ctx.prove_fs_packed_async(3, pin, out, cu)
    ctx.verify_fs_packed_async(3, out, res)
    assert np.array_equal(out, ro) and np.array_equal(cu, rc) and np.array_equal(res, rr)
    with pytest.raises(P.PbhError):
        ctx.prove_fs_packed_async(4, pin, out)
    for b, _, _ in sets:
        for arr in b.values():
            ctx.host_free(arr)


@pytest.mark.gpu
def test_fs_packed_guard_bytes_and_arguments(gpu_ctx, oracle):
    """12-byte records at 4- but not 16-byte-aligned device addresses leave the bytes around them untouched; n = 0 is a no-op;
    null and misaligned pointers are refused."""
    import torch
    import pbh_b200 as P
    ctx = gpu_ctx["table"]
    lib = ctx.lib
    dev = torch.device("cuda", 0)
    n = 1001
    w, r, want, want_cu, vo, _ = _expect(oracle, 255, P.DIST_FULLPATH)
    w, r = np.tile(w, 4)[:, :n].copy(), np.tile(r, 4)[:, :n].copy()
    want, want_cu, vo = np.tile(want, (4, 1))[:n], np.tile(want_cu, 4)[:n], np.tile(vo, 4)[:n]
    pin = P.pack_fs_witness(w, r)
    g = 36
    big = lambda nbytes: torch.full((nbytes + 2 * g,), 0xAB, dtype=torch.uint8, device=dev)
    IN, OUT, CU, RES = big(12 * n), big(12 * n), big(4 * n), big(n)
    for off in (4, 20):
        IN[:] = 0xAB
        IN[off:off + 12 * n] = torch.from_numpy(pin.view(np.uint8)).to(dev)
        OUT[:] = 0xAB; CU[:] = 0xAB; RES[:] = 0xAB
        views = [t[off:off + k * n] for t, k in ((IN, 12), (OUT, 12), (CU, 4))]
        assert all(v.data_ptr() % 4 == 0 and v.data_ptr() % 16 != 0 for v in views)
        ctx.prove_fs_packed(views[0], out=views[1], chal_u=views[2])
        ctx.verify_fs_packed(views[1], result=RES[off + 1:off + 1 + n])
        ctx.sync()
        assert np.array_equal(views[1].cpu().numpy().view("<u4").reshape(-1, 3), want)
        assert np.array_equal(views[2].cpu().numpy().view("<u4"), want_cu)
        assert np.array_equal(RES[off + 1:off + 1 + n].cpu().numpy(), vo)
        for t, k, o in ((OUT, 12, off), (CU, 4, off), (RES, 1, off + 1)):
            assert bool((t[:o] == 0xAB).all()) and bool((t[o + k * n:] == 0xAB).all())
    h, p = ctx.h, lambda t: C.c_void_p(t.data_ptr())
    host = np.zeros(16 * n, np.uint8); hp = C.c_void_p(host.ctypes.data)
    launches = ctx.launch_count
    # n = 0: nothing happens, whatever the pointers
    assert lib.pbh_prove_fs_packed_dev(h, C.c_size_t(0), None, None, None) == 0
    assert lib.pbh_verify_fs_packed_dev(h, C.c_size_t(0), None, None) == 0
    assert lib.pbh_prove_fs_packed(h, C.c_size_t(0), None, None, None) == 0
    assert lib.pbh_verify_fs_packed(h, C.c_size_t(0), None, None) == 0
    assert lib.pbh_prove_fs_packed_async(h, 0, C.c_size_t(0), None, None, None) == 0
    assert lib.pbh_verify_fs_packed_async(h, 0, C.c_size_t(0), None, None) == 0
    assert ctx.launch_count == launches
    # null pointers
    assert lib.pbh_prove_fs_packed_dev(h, C.c_size_t(n), None, p(OUT), None) == -1
    assert lib.pbh_prove_fs_packed_dev(h, C.c_size_t(n), p(IN), None, None) == -1
    assert lib.pbh_verify_fs_packed_dev(h, C.c_size_t(n), None, p(RES)) == -1
    assert lib.pbh_verify_fs_packed_dev(h, C.c_size_t(n), p(OUT), None) == -1
    assert lib.pbh_prove_fs_packed(h, C.c_size_t(n), hp, None, None) == -1
    assert lib.pbh_verify_fs_packed(h, C.c_size_t(n), None, hp) == -1
    assert lib.pbh_prove_fs_packed_async(h, 1, C.c_size_t(n), None, hp, None) == -1
    assert lib.pbh_verify_fs_packed_async(h, 1, C.c_size_t(n), hp, None) == -1
    assert lib.pbh_verify_fs_packed_async(h, -1, C.c_size_t(n), hp, hp) == -1
    # device records that are not 4-byte aligned
    mis = lambda t: C.c_void_p(t.data_ptr() + 2)
    assert lib.pbh_prove_fs_packed_dev(h, C.c_size_t(n), mis(IN), p(OUT), None) == -1
    assert lib.pbh_prove_fs_packed_dev(h, C.c_size_t(n), p(IN), mis(OUT), None) == -1
    assert lib.pbh_prove_fs_packed_dev(h, C.c_size_t(n), p(IN), p(OUT), mis(CU)) == -1
    assert lib.pbh_verify_fs_packed_dev(h, C.c_size_t(n), mis(OUT), p(RES)) == -1
    assert ctx.launch_count == launches
    with pytest.raises(P.PbhError):
        ctx.prove_fs_packed(IN[2:2 + 12 * n])
    ctx.sync()
