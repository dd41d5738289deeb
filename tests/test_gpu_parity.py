"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle — bit-exact.

Mirrors the reference's own tests where it has them (src/pbh/mod.rs:44-124 end to end, src/pbh/g1.rs:233-260,
src/pbh/gt.rs:88-97, src/pbh/pairing.rs:56-75, src/fft.rs:140-183, src/poly.rs:428-434) and adds what SURVEY.md §4 asks
for: exhaustive small domains, seeded batches over every status class, adversarial verifier inputs and
size-independent properties at BASELINE.json's batch sizes.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ALGOS = ("table", "arith")
CTXS = ("table", "table_generic", "table_notma", "table_int", "table_vf32", "arith", "arith_int")   # gpu_ctx keys: table = FP32-pipe prover with TMA tiles (default),
# table_generic = same without the compile-time circuit constants, table_notma = plain loads/stores, table_int = int32
# prover and verifier, table_vf32 = verifier scalars on the FP32 pipes, arith = per-item curve arithmetic (FP32 core),
# arith_int = per-item curve arithmetic (int32 prover)


def _np(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)


# ---------------------------------------------------------------------------------------------
# the reference's only end-to-end test, written the way the reference writes it (src/pbh/mod.rs:44-124)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ALGOS)
def test_plonk_gen_proof(product_lib, algo):
    from pbh_b200 import (SRS, Assigment, Assigments, Challange, Constrains, CopyOf, Gate, Plonk, Proof, f17, f101, g1f)

    s = f101(2)
    srs = SRS.create(s, 6)
    plonk = Plonk.new(srs, f17(4), algo=algo)
    constraints = Constrains(
        [Gate.mul_a_b(), Gate.mul_a_b(), Gate.mul_a_b(), Gate.sum_a_b()],
        ([CopyOf.B(1), CopyOf.B(2), CopyOf.B(3), CopyOf.C(1)],
         [CopyOf.A(1), CopyOf.A(2), CopyOf.A(3), CopyOf.C(2)],
         [CopyOf.A(4), CopyOf.B(4), CopyOf.C(4), CopyOf.C(3)]))
    assigments = Assigments([Assigment(f17(3), f17(3), f17(9)), Assigment(f17(4), f17(4), f17(16)),
                             Assigment(f17(5), f17(5), f17(25)), Assigment(f17(9), f17(16), f17(25))])
    rand = [f17(7), f17(4), f17(11), f17(12), f17(16), f17(2), f17(14), f17(11), f17(7)]
    challange = Challange(alpha=f17(15), beta=f17(12), gamma=f17(13), z=f17(5), v=f17(12))

    proof = plonk.prove(constraints, assigments, challange, rand)
    expected = Proof(a_s=g1f(91, 66), b_s=g1f(26, 45), c_s=g1f(91, 35), z_s=g1f(32, 59), t_lo_s=g1f(12, 32),
                     t_mid_s=g1f(26, 45), t_hi_s=g1f(91, 66), w_z_s=g1f(91, 35), w_z_omega_s=g1f(65, 98), a_z=f17(15),
                     b_z=f17(13), c_z=f17(5), s_sigma_1_z=f17(1), s_sigma_2_z=f17(12), r_z=f17(15), z_omega_z=f17(15))
    assert proof == expected
    rand = [f17(4)]
    assert plonk.verify(constraints, proof, challange, rand)


@pytest.mark.parametrize("algo", ALGOS)
def test_golden_pairing_value_93_76u(gpu_ctx, oracle, algo):
    """README.md:6 of the reference: the pairing of the golden proof is 93+76u (not the tutorial's 97+89u)."""
    ctx = gpu_ctx[algo]
    wit = np.array([[3, 4, 5, 9, 3, 4, 5, 16, 9, 16, 8, 8]], dtype=np.uint8).T.copy()
    rnd = np.array([[7, 4, 11, 12, 16, 2, 14, 11, 7]], dtype=np.uint8).T.copy()
    chal = np.array([[15, 12, 13, 5, 12]], dtype=np.uint8).T.copy()
    proof, status = ctx.prove_batch(wit, rnd, chal)
    assert status.tolist() == [0]
    res, gt = ctx.verify_batch(proof, chal, np.array([4], dtype=np.uint8), want_gt=True)
    assert res.tolist() == [1] and gt[:, 0].tolist() == [93, 76, 93, 76]


def test_reference_panics_surface_as_exceptions(product_lib):
    """SURVEY.md §9: (4,4,7) | 0,0,10,0,7,0,0,0,16 | 7,4,2,16,16 makes prove panic at src/plonk.rs:370 (Q1)."""
    from pbh_b200 import (SRS, Assigment, Assigments, Challange, Constrains, CopyOf, Gate, Plonk, ReferencePanic)
    plonk = Plonk.new(SRS.create(2, 6), 4)
    constraints = Constrains([Gate.mul_a_b()] * 3 + [Gate.sum_a_b()],
                             ([CopyOf.B(1), CopyOf.B(2), CopyOf.B(3), CopyOf.C(1)], [CopyOf.A(1), CopyOf.A(2), CopyOf.A(3), CopyOf.C(2)],
                              [CopyOf.A(4), CopyOf.B(4), CopyOf.C(4), CopyOf.C(3)]))
    x, y, z = 4, 4, 7
    ass = Assigments([Assigment(x, x, x * x), Assigment(y, y, y * y), Assigment(z, z, z * z), Assigment(x * x, y * y, z * z)])
    with pytest.raises(ReferencePanic) as e:
        plonk.prove(constraints, ass, Challange(7, 4, 2, 16, 16), [0, 0, 10, 0, 7, 0, 0, 0, 16])
    assert e.value.status == 3
    # an unsatisfied witness panics at src/plonk.rs:199
    bad = Assigments([Assigment(3, 3, 9), Assigment(4, 4, 16), Assigment(5, 5, 25), Assigment(9, 16, 24)])
    with pytest.raises(ReferencePanic) as e:
        plonk.prove(constraints, bad, Challange(15, 12, 13, 5, 12), [7, 4, 11, 12, 16, 2, 14, 11, 7])
    assert e.value.status == 1


# ---------------------------------------------------------------------------------------------
# seeded batches, every status class, both distributions, both algorithms
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", CTXS)
@pytest.mark.parametrize("dist", (0, 1))
def test_prove_verify_batches_match_oracle(gpu_ctx, oracle, algo, dist):
    ctx = gpu_ctx[algo]
    n = 30000 + 37          # ragged: not a multiple of the block or vector width
    w, r, c, u, att = ctx.generate_inputs(n, first_index=1000, seed=0xB200 + dist, dist=dist, want_attempt=True)
    wo, ro, co, uo, atto = oracle.generate_inputs(n, first_index=1000, seed=0xB200 + dist, dist=dist, threads=8)
    assert np.array_equal(_np(w), wo) and np.array_equal(_np(r), ro) and np.array_equal(_np(c), co)
    assert np.array_equal(_np(u), uo) and np.array_equal(_np(att), atto)

    proof, status = ctx.prove_batch(w, r, c)
    res, gt = ctx.verify_batch(proof, c, u, want_gt=True)
    ctx.sync()
    po, so = oracle.prove_batch(wo, ro, co, threads=8)
    vo, go = oracle.verify_batch(po, co, uo, threads=8)
    assert np.array_equal(_np(status), so)
    assert np.array_equal(_np(proof), po)
    assert np.array_equal(_np(res), vo)
    assert np.array_equal(_np(gt), go)
    if dist == 0:
        # every class of SURVEY.md §2.4 is present in a uniform batch of this size
        assert set(np.unique(so)) >= {0, 2, 4, 5}
        assert set(np.unique(vo)) >= {0, 1, 2, 0x10}
    else:
        assert (so == 0).all() and set(np.unique(vo)) == {0, 1}

    # host-pointer entry points: same bytes
    ph, sh = ctx.prove_batch(wo, ro, co)
    vh, gh = ctx.verify_batch(po, co, uo, want_gt=True)
    assert np.array_equal(ph, po) and np.array_equal(sh, so) and np.array_equal(vh, vo) and np.array_equal(gh, go)


def test_extra_end_to_end_tuples(gpu_ctx, oracle):
    """The derived tuples of SURVEY.md §9 (true / false / identity pairing 0+0u / in_curve false / Z_H panic / Q1 panic)."""
    rows = [
        ((9, 15, 0), (14, 11, 11, 2, 7, 3, 7, 15, 6), (10, 6, 15, 0, 15), 11, 0, 1, (7, 28, 7, 28)),
        ((7, 0, 10), (13, 5, 1, 2, 12, 16, 9, 7, 9), (1, 14, 5, 5, 8), 14, 0, 1, (2, 7, 2, 7)),
        ((0, 16, 1), (15, 8, 11, 4, 16, 16, 6, 2, 8), (7, 12, 12, 14, 13), 9, 0, 1, (31, 96, 31, 96)),
        ((0, 1, 16), (3, 11, 4, 0, 15, 12, 10, 2, 15), (9, 0, 3, 15, 11), 6, 0, 0, (38, 95, 2, 7)),
        ((15, 3, 9), (1, 2, 4, 0, 7, 1, 6, 6, 15), (5, 0, 12, 3, 16), 12, 0, 0, (26, 97, 0, 0)),
        ((0, 6, 11), (7, 13, 10, 13, 8, 1, 14, 8, 14), (14, 11, 7, 10, 10), 2, 0, 1, (0, 0, 0, 0)),
        ((5, 3, 0), (11, 15, 9, 2, 13, 5, 16, 13, 9), (8, 0, 6, 5, 14), 5, 0, 2, (0, 0, 0, 0)),
        ((4, 3, 12), (9, 10, 6, 6, 5, 6, 12, 9, 0), (11, 13, 5, 4, 8), 2, 0, 0x10, (0, 0, 0, 0)),
        ((4, 4, 7), (0, 0, 10, 0, 7, 0, 0, 0, 16), (7, 4, 2, 16, 16), 0, 3, None, None),
    ]
    n = len(rows)
    wit = np.zeros((12, n), np.uint8); rnd = np.zeros((9, n), np.uint8); chal = np.zeros((5, n), np.uint8); u = np.zeros(n, np.uint8)
    for i, ((x, y, z), r, c, uu, *_rest) in enumerate(rows):
        xx, yy, zz = x * x % 17, y * y % 17, z * z % 17
        wit[:, i] = [x, y, z, xx, x, y, z, yy, xx, yy, zz, zz]
        rnd[:, i] = r; chal[:, i] = c; u[i] = uu
    for algo in CTXS:
        ctx = gpu_ctx[algo]
        proof, status = ctx.prove_batch(wit, rnd, chal)
        assert status.tolist() == [row[4] for row in rows]
        res, gt = ctx.verify_batch(proof, chal, u, want_gt=True)
        for i, row in enumerate(rows):
            if row[5] is not None:
                assert int(res[i]) == row[5], (algo, i)
                assert tuple(int(v) for v in gt[:, i]) == row[6], (algo, i)
    po, so = oracle.prove_batch(wit, rnd, chal)
    assert so.tolist() == [row[4] for row in rows]


# ---------------------------------------------------------------------------------------------
# adversarial verifier inputs (SURVEY.md §4 iv)
# ---------------------------------------------------------------------------------------------
def _tamper(proof, chal, u, rng):
    """Flip bytes of honest proofs: non-subgroup and off-curve points, identity flags with coordinates, evaluations
    outside F_17, coordinates outside F_101, challenges in H."""
    p = proof.copy(); c = chal.copy(); uu = u.copy()
    n = p.shape[1]
    curve = np.array([(x, y) for x in range(101) for y in range(101) if (y * y - x * x * x - 3) % 101 == 0], dtype=np.uint8)
    kind = rng.integers(0, 10, size=n)
    for i in range(n):
        k = kind[i]
        pt = rng.integers(0, 9)
        if k == 0:      # any curve point (Q17: mostly outside the order-17 subgroup)
            p[2 * pt:2 * pt + 2, i] = curve[rng.integers(0, len(curve))]
        elif k == 1:    # random coordinates (mostly off-curve)
            p[2 * pt:2 * pt + 2, i] = rng.integers(0, 101, size=2)
        elif k == 2:    # infinity flag on a point that keeps its coordinates: passes in_curve, acts as identity
            if pt < 8: p[18, i] |= 1 << pt
            else: p[19, i] |= 1
        elif k == 3:    # canonical identity (0,0,inf): fails in_curve (Q9)
            p[2 * pt:2 * pt + 2, i] = 0
            if pt < 8: p[18, i] |= 1 << pt
            else: p[19, i] |= 1
        elif k == 4:    # tampered evaluation, in the field
            p[20 + rng.integers(0, 7), i] = rng.integers(0, 17)
        elif k == 5:    # evaluation outside the field
            p[20 + rng.integers(0, 7), i] = rng.integers(17, 256)
        elif k == 6:    # coordinate byte outside F_101 / stray flag bits / challenge byte outside F_17
            j = rng.integers(0, 4)
            if j == 0: p[rng.integers(0, 18), i] = rng.integers(101, 256)
            elif j == 1: p[19, i] |= 1 << rng.integers(1, 8)
            elif j == 2: c[rng.integers(0, 5), i] = rng.integers(17, 256)
            else: uu[i] = rng.integers(17, 256)
        elif k == 7:    # z in H: Z_H(z) = 0 (Q4)
            c[3, i] = [1, 4, 13, 16][rng.integers(0, 4)]
        elif k == 8:    # several curve points at once, including order-2 / order-3 / order-6 points
            for q in rng.integers(0, 9, size=3):
                p[2 * q:2 * q + 2, i] = curve[rng.integers(0, len(curve))]
        # k == 9: untouched
    return p, c, uu


@pytest.mark.parametrize("algo", ALGOS)
def test_verify_adversarial_inputs(gpu_ctx, oracle, algo):
    ctx = gpu_ctx[algo]
    n = 40000
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=77, dist=1, threads=8)
    po, so = oracle.prove_batch(wo, ro, co, threads=8)
    assert (so == 0).all()
    p, c, u = _tamper(po, co, uo, np.random.default_rng(5))
    vo, go = oracle.verify_batch(p, c, u, threads=8)
    res, gt = ctx.verify_batch(p, c, u, want_gt=True)
    assert np.array_equal(res, vo)
    assert np.array_equal(gt, go)
    assert set(np.unique(vo)) >= {0, 1, 2, 4, 0x10, 0x20}


@pytest.mark.parametrize("algo", CTXS)
def test_zero_blinder_corner_cases(gpu_ctx, oracle, algo):
    """Blinders and challenges drawn from a few values with many zeros: short polynomials, the Q1 / Q5 / Q15 length
    logic, and the hand-over between the FP32 fast path and the exact integer routine."""
    rng = np.random.default_rng(17)
    n = 60000
    w = oracle.generate_inputs(n, seed=5, dist=0, threads=8)[0]
    r = rng.choice(np.array([0, 0, 0, 1, 16, 5], dtype=np.uint8), size=(9, n))
    c = rng.choice(np.array([0, 1, 16, 3, 7], dtype=np.uint8), size=(5, n))
    po, so = oracle.prove_batch(w, r, c, threads=8)
    p, s = gpu_ctx[algo].prove_batch(w, r, c)
    assert np.array_equal(s, so) and np.array_equal(p, po)
    assert (so == 3).sum() > 0 and (so == 4).sum() > 0 and (so == 0).sum() > 0


def test_prove_bad_encoding(gpu_ctx, oracle):
    n = 512
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=3, dist=1)
    wo[5, 7] = 17; ro[0, 9] = 200; co[4, 11] = 255
    po, so = oracle.prove_batch(wo, ro, co)
    for algo in CTXS:
        p, s = gpu_ctx[algo].prove_batch(wo, ro, co)
        assert np.array_equal(s, so) and np.array_equal(p, po)
    assert so[7] == 32 and so[9] == 32 and so[11] == 32


# ---------------------------------------------------------------------------------------------
# other circuits and SRS parameters (generic 4-gate circuits; Q11; longer SRS removes the Q2 panic)
# ---------------------------------------------------------------------------------------------
def test_other_circuits_and_srs(product_lib, oracle):
    import pbh_b200
    rng = np.random.default_rng(11)
    n = 4000
    cases = [dict(s=2, srs_n=6), dict(s=3, srs_n=6), dict(s=7, srs_n=9), dict(s=100, srs_n=8), dict(s=2, srs_n=4), dict(s=55, srs_n=12)]
    for case in cases:
        # pbh circuit with uniform inputs, then a randomised circuit (random selectors and copy constraints)
        for randomise in (False, "qc0", "full"):
            oc = oracle.pbh_test_circuit(); pc = pbh_b200.pbh_test_circuit()
            if randomise:
                for name in ("q_l", "q_r", "q_o", "q_m", "q_c"):
                    vals = rng.integers(0, 17, size=4)
                    if name == "q_c" and randomise == "qc0":
                        vals[:] = 0      # then the zero witness satisfies the circuit and the deeper sites are reached
                    for i in range(4):
                        getattr(oc, name)[i] = int(vals[i]); getattr(pc, name)[i] = int(vals[i])
                for name in ("c_a", "c_b", "c_c"):
                    ws = rng.integers(0, 3, size=4); idx = rng.integers(1, 5, size=4)
                    for i in range(4):
                        getattr(oc, name + "_wire")[i] = int(ws[i]); getattr(pc, name + "_wire")[i] = int(ws[i])
                        getattr(oc, name + "_index")[i] = int(idx[i]); getattr(pc, name + "_index")[i] = int(idx[i])
            wit = rng.integers(0, 17, size=(12, n), dtype=np.uint8)
            if not randomise:
                wit = oracle.generate_inputs(n, seed=int(rng.integers(1 << 30)), dist=0)[0]
            else:
                wit[:, : n // 2] = wit[:, :1]   # constant witnesses satisfy copy constraints more often
                wit[:, : n // 4] = 0            # the zero witness satisfies any circuit with q_c = 0
            rnd = rng.integers(0, 17, size=(9, n), dtype=np.uint8)
            chal = rng.integers(0, 17, size=(5, n), dtype=np.uint8)
            u = rng.integers(0, 17, size=n, dtype=np.uint8)
            po, so = oracle.prove_batch(wit, rnd, chal, circuit=oc, threads=8, **case)
            vo, go = oracle.verify_batch(po, chal, u, circuit=oc, threads=8, **case)
            for algo in CTXS:
                with pbh_b200.Context(circuit=pc, device=0, algo=algo.split("_")[0], **case) as ctx:
                    if algo.endswith("_int"):
                        ctx.set_option(pbh_b200.OPT_PROVER_FP32, 0)
                    if algo.endswith("_notma"):
                        ctx.set_option(pbh_b200.OPT_TMA, 0)
                    g1s, g2 = ctx.srs()
                    og1s, og2, oconst = oracle.setup(circuit=oc, **case)
                    assert np.array_equal(g1s, og1s) and np.array_equal(g2, og2)
                    assert np.array_equal(ctx.verifier_constants(), oconst)
                    p, s = ctx.prove_batch(wit, rnd, chal)
                    assert np.array_equal(s, so), (case, randomise, algo)
                    assert np.array_equal(p, po), (case, randomise, algo)
                    v, g = ctx.verify_batch(po, chal, u, want_gt=True)
                    assert np.array_equal(v, vo) and np.array_equal(g, go), (case, randomise, algo)


def test_setup_panics_match_reference(product_lib, oracle):
    """SRS::create panics for s = 0 and for every s whose double-and-add hits P + (-P) in G2 (Q12)."""
    import pbh_b200
    for s in range(101):
        try:
            oracle.setup(s=s)
            o_ok = True
        except ArithmeticError:
            o_ok = False
        try:
            pbh_b200.Context(s=s, device=0).close()
            p_ok = True
        except pbh_b200.ReferencePanic:
            p_ok = False
        assert o_ok == p_ok, s
    assert not o_ok or True


# ---------------------------------------------------------------------------------------------
# sweep kernels: exhaustive small domains
# ---------------------------------------------------------------------------------------------
def test_ntt4_intt4_exhaustive(gpu_ctx, oracle):
    """All 17^4 inputs: interpolate_at_h (src/plonk.rs:177-179) == size-4 iNTT, and NTT(iNTT(v)) == v."""
    ctx = gpu_ctx["table"]
    g = np.arange(17, dtype=np.uint8)
    v = np.stack(np.meshgrid(g, g, g, g, indexing="ij")).reshape(4, -1)
    # host planes are staged with pitch n: 83521 and 83518 take the byte loop, 83536 (padded with zeros) the 128-bit path
    for arr in (v, v[:, :83521 - 3], np.pad(v, ((0, 0), (0, 83536 - 83521)))):
        arr = np.ascontiguousarray(arr)
        c = ctx.intt4_batch(arr)
        assert np.array_equal(c, oracle.intt4_batch(arr))
        e = ctx.ntt4_batch(c)
        assert np.array_equal(e, arr)
        assert np.array_equal(ctx.ntt4_batch(arr), oracle.ntt4_batch(arr))


def test_ntt_generic_reference_vectors(gpu_ctx, oracle):
    """src/fft.rs:140-183: F_337, omega = 85, n = 8."""
    ctx = gpu_ctx["table"]
    vals = np.array([[3, 1, 4, 1, 5, 9, 2, 6]], dtype=np.uint16).T.copy()
    freq = ctx.ntt_generic_batch(vals, 337, 85)
    assert freq[:, 0].tolist() == [31, 70, 109, 74, 334, 181, 232, 4]
    assert ctx.ntt_generic_batch(freq, 337, 85, inverse=True)[:, 0].tolist() == [3, 1, 4, 1, 5, 9, 2, 6]
    # NTT product of [24,12,28,8] and [4,26,29,23] equals the schoolbook product (src/fft.rs:171-183)
    a = np.array([[24, 12, 28, 8, 0, 0, 0, 0]], dtype=np.uint16).T.copy(); b = np.array([[4, 26, 29, 23, 0, 0, 0, 0]], dtype=np.uint16).T.copy()
    fa, fb = ctx.ntt_generic_batch(a, 337, 85), ctx.ntt_generic_batch(b, 337, 85)
    prod = ((fa.astype(np.uint32) * fb) % 337).astype(np.uint16)
    assert ctx.ntt_generic_batch(prod, 337, 85, inverse=True)[:, 0].tolist() == [96, 335, 109, 312, 285, 202, 184, 0]
    # random batches against the oracle's CooleyTurkey, sizes 2..64 over F_337 (omega = 85 has order 8) and F_257 (3 has order 256)
    rng = np.random.default_rng(2)
    for mod, root, order in ((337, 85, 8), (257, 3, 256)):
        for size in (2, 4, 8, 16, 32, 64):
            if size > order:
                continue
            omega = pow(root, order // size, mod)
            x = rng.integers(0, mod, size=(size, 300)).astype(np.uint16)
            for inverse in (False, True):
                got = ctx.ntt_generic_batch(x, mod, omega, inverse=inverse)
                for j in range(0, 300, 37):
                    exp = oracle.fft(mod, omega, size, "cooley_tukey", inverse, x[:, j].tolist())
                    assert got[:, j].tolist() == exp, (mod, size, inverse, j)


def test_g1_add_smul_exhaustive(gpu_ctx, oracle):
    """All 102 x 102 additions and 102 x 101 scalar multiples of the curve group, identity included, plus flagged
    points that keep coordinates and off-curve operands (src/pbh/g1.rs:119-168, vectors of :233-260)."""
    ctx = gpu_ctx["arith"]
    pts = [(x, y, 0) for x in range(101) for y in range(101) if (y * y - x * x * x - 3) % 101 == 0] + [(0, 0, 1)]
    assert len(pts) == 102
    P = np.array(pts, dtype=np.uint8)
    a = np.repeat(P, 102, axis=0); b = np.tile(P, (102, 1))
    arr = np.ascontiguousarray(np.concatenate([a, b], axis=1).T)
    assert np.array_equal(ctx.g1_add_batch(arr), oracle.g1_add_batch(arr))
    sm = np.ascontiguousarray(np.concatenate([np.repeat(P, 101, axis=0), np.tile(np.arange(101, dtype=np.uint8), 102)[:, None]], axis=1).T)
    got = ctx.g1_smul_batch(sm)
    assert np.array_equal(got, oracle.g1_smul_batch(sm))
    # reference vectors: 2G, 4G, 8G, 16G, 3G, 5G, 9G
    G = (1, 2, 0)
    for k, exp in ((2, (68, 74)), (4, (65, 98)), (8, (18, 49)), (16, (1, 99)), (3, (26, 45)), (5, (12, 32)), (9, (18, 52)), (17, None)):
        o = ctx.g1_smul_batch(np.array([[G[0]], [G[1]], [0], [k]], dtype=np.uint8))[:, 0].tolist()
        assert o == ([exp[0], exp[1], 0] if exp else [0, 0, 1])
    # random operands incl. off-curve points and flagged points with coordinates
    rng = np.random.default_rng(8)
    r = rng.integers(0, 101, size=(6, 20000), dtype=np.uint8)
    r[2] = rng.integers(0, 2, size=20000); r[5] = rng.integers(0, 2, size=20000)
    assert np.array_equal(ctx.g1_add_batch(r), oracle.g1_add_batch(r))
    r4 = rng.integers(0, 101, size=(4, 20000), dtype=np.uint8); r4[2] = rng.integers(0, 2, size=20000)
    on = rng.integers(0, 101, size=20000)
    r4[0, :10000] = P[on[:10000], 0]; r4[1, :10000] = P[on[:10000], 1]
    assert np.array_equal(ctx.g1_smul_batch(r4), oracle.g1_smul_batch(r4))


def test_pairing_exhaustive(gpu_ctx, oracle):
    """Every curve point (and the identity, and flagged points) against every multiple of the G2 generator:
    Miller loop + final exponentiation (src/pbh/pairing.rs:12-47); bilinearity as in src/pbh/pairing.rs:56-75."""
    ctx = gpu_ctx["arith"]
    pts = [(x, y, 0) for x in range(101) for y in range(101) if (y * y - x * x * x - 3) % 101 == 0] + [(0, 0, 1), (1, 2, 1), (48, 0, 1)]
    g2 = [oracle.g2_mul((36, 31), k) for k in range(1, 17)]
    rows = [(p[0], p[1], p[2], q[0], q[1]) for p in pts for q in g2]
    arr = np.ascontiguousarray(np.array(rows, dtype=np.uint8).T)
    got = ctx.pairing_batch(arr)
    exp = oracle.pairing_batch(arr)
    assert np.array_equal(got, exp)
    # the values the survey derived: e(G, G2) = 7+28u, e(2G, G2) = 97+89u, e(12G, G2) = 93+76u, e(inf, .) = 0+0u
    lut = {(r[0], r[1], r[2], r[3], r[4]): tuple(int(v) for v in got[:, i]) for i, r in enumerate(rows)}
    assert lut[(1, 2, 0, 36, 31)] == (7, 28) and lut[(68, 74, 0, 36, 31)] == (97, 89) and lut[(12, 69, 0, 36, 31)] == (93, 76)
    assert lut[(0, 0, 1, 36, 31)] == (0, 0) and lut[(6, 44, 0, 36, 31)] == (31, 5) and lut[(48, 0, 0, 36, 31)] == (0, 0)
    # arbitrary (a, b) second arguments, not only G2 multiples
    rng = np.random.default_rng(4)
    r = rng.integers(0, 101, size=(5, 30000), dtype=np.uint8); r[2] = rng.integers(0, 2, size=30000)
    sel = rng.integers(0, 102, size=30000)
    P = np.array(pts[:102], dtype=np.uint8)
    r[0] = P[sel, 0]; r[1] = P[sel, 1]
    assert np.array_equal(ctx.pairing_batch(r), oracle.pairing_batch(r))


@pytest.mark.parametrize("algo", ALGOS)
def test_kzg_commit_sweep(gpu_ctx, oracle, algo):
    """SRS::eval_at_s over random 7-coefficient polynomials (src/plonk.rs:51-58)."""
    ctx = gpu_ctx[algo]
    rng = np.random.default_rng(6)
    c = rng.integers(0, 17, size=(7, 50001), dtype=np.uint8)
    c[:, :17] = 0
    c[0, :17] = np.arange(17)
    assert np.array_equal(ctx.kzg_commit_batch(c), oracle.kzg_commit_batch(c))
    # any byte value is a coefficient (F17::from reduces it); device pointers; sizes around the 4-items-per-word path
    import torch
    for n in (1, 3, 4, 7, 4096, 20003):
        c = rng.integers(0, 256, size=(7, n), dtype=np.uint8)
        exp = oracle.kzg_commit_batch(c)
        assert np.array_equal(ctx.kzg_commit_batch(c), exp), n
        got = ctx.kzg_commit_batch(torch.from_numpy(c).cuda())
        ctx.sync()
        assert np.array_equal(got.cpu().numpy(), exp), n


def test_poly_sweeps(gpu_ctx, oracle):
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(9)
    n = 20011
    # src/poly.rs:428-434 over F_17: [5,0,10,6] * [1,2,4]
    a = np.array([[5, 0, 10, 6]], dtype=np.uint8).T.copy(); b = np.array([[1, 2, 4]], dtype=np.uint8).T.copy()
    assert ctx.poly_mul_batch(a, b)[:, 0].tolist() == [v % 17 for v in [5, 10, 30, 26, 52, 24]]
    for la, lb in ((1, 1), (2, 5), (4, 4), (6, 6), (7, 4), (11, 6), (16, 7), (16, 16)):
        a = rng.integers(0, 17, size=(la, n), dtype=np.uint8); b = rng.integers(0, 17, size=(lb, n), dtype=np.uint8)
        a[:, : n // 8] = 0
        assert np.array_equal(ctx.poly_mul_batch(a, b), oracle.poly_mul_batch(a, b)), (la, lb)
    for ln in (1, 4, 22):
        a = rng.integers(0, 17, size=(ln, n), dtype=np.uint8); b = rng.integers(0, 17, size=(ln, n), dtype=np.uint8)
        assert np.array_equal(ctx.poly_add_batch(a, b), oracle.poly_add_batch(a, b))
        assert np.array_equal(ctx.poly_add_batch(a, b, subtract=True), oracle.poly_add_batch(a, b, subtract=True))
    p = rng.integers(0, 17, size=(22, n), dtype=np.uint8)
    p[18:, : n // 4] = 0; p[:, : n // 16] = 0
    q, r = ctx.poly_div_zh_batch(p)
    qo, ro = oracle.poly_div_zh_batch(p)
    assert np.array_equal(q, qo) and np.array_equal(r, ro)


def test_poly_scale_eval_div_linear_sweeps(gpu_ctx, oracle):
    """Poly * scalar (src/poly.rs:220-228), Poly::eval (:71-79), Poly / (x - c) (:230-247), host and device pointers,
    word-aligned and ragged sizes, non-canonical bytes reduced as F17::from does."""
    import torch
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(11)
    # src/poly.rs tests: eval of 1 + 2x + 3x^2 at 2 is 17 = 0 mod 17
    assert ctx.poly_eval_batch(np.array([[1, 2, 3, 2]], dtype=np.uint8).T.copy())[0] == 0
    for n in (1, 3, 4096, 20011):
        for ln in (1, 2, 7, 10, 22):
            arr = rng.integers(0, 17, size=(ln + 1, n), dtype=np.uint8)
            arr[ln, : n // 5] = 0                       # scale by 0 (Q15), evaluate at 0, divide by x
            arr[:, n // 2: n // 2 + n // 7] = rng.integers(0, 256, size=(ln + 1, n // 7), dtype=np.uint8)
            so, eo, do = oracle.poly_scale_batch(arr), oracle.poly_eval_batch(arr), oracle.poly_div_linear_batch(arr)
            assert np.array_equal(ctx.poly_scale_batch(arr), so), (n, ln)
            assert np.array_equal(ctx.poly_eval_batch(arr), eo), (n, ln)
            assert np.array_equal(ctx.poly_div_linear_batch(arr), do), (n, ln)
            assert np.array_equal(do[ln - 1], eo)       # remainder theorem
            if n > 1000:
                d = torch.from_numpy(arr).cuda()
                got = [ctx.poly_scale_batch(d), ctx.poly_eval_batch(d), ctx.poly_div_linear_batch(d)]
                ctx.sync()
                assert np.array_equal(got[0].cpu().numpy(), so) and np.array_equal(got[1].cpu().numpy(), eo) and np.array_equal(got[2].cpu().numpy(), do)


def test_mul_ntt_sweep(gpu_ctx, oracle):
    """mul_ntt (src/fft.rs:109-132): the reference's own vector (src/fft.rs:171-183) and random batches against the
    oracle's CooleyTurkey restatement over F_337 and F_257."""
    ctx = gpu_ctx["table"]
    a = np.array([[24, 12, 28, 8]], dtype=np.uint16).T.copy(); b = np.array([[4, 26, 29, 23]], dtype=np.uint16).T.copy()
    assert ctx.mul_ntt_batch(a, b, 337, 85)[:, 0].tolist() == [96, 335, 109, 312, 285, 202, 184, 0]
    rng = np.random.default_rng(4)
    for mod, root, order in ((337, 85, 8), (257, 3, 256)):
        for la, lb in ((1, 1), (2, 2), (3, 5), (4, 4), (7, 9), (16, 16), (40, 24)):
            size = la + lb
            if size > order:
                continue
            omega = pow(root, order // size, mod)
            x = rng.integers(0, mod, size=(la, 2000)).astype(np.uint16); y = rng.integers(0, mod, size=(lb, 2000)).astype(np.uint16)
            assert np.array_equal(ctx.mul_ntt_batch(x, y, mod, omega), oracle.mul_ntt_batch(x, y, mod, omega)), (mod, la, lb)


# ---------------------------------------------------------------------------------------------
# layout: pitches, sub-ranges, empty batches; shard summaries
# ---------------------------------------------------------------------------------------------
def test_pitch_subranges_and_empty(gpu_ctx, oracle):
    import torch
    ctx = gpu_ctx["table"]
    N, lo, hi = 5000, 1237, 4096
    wo, ro, co, uo, _ = oracle.generate_inputs(N, seed=21, dist=0)
    po, so = oracle.prove_batch(wo, ro, co)
    # host: column slices of a larger batch are addressed through the pitch, without repacking
    proof = np.zeros((27, N), np.uint8); status = np.full(N, 0xEE, np.uint8)
    ctx.prove_batch(wo[:, lo:hi], ro[:, lo:hi], co[:, lo:hi], proof=proof[:, lo:hi], status=status[lo:hi])
    assert np.array_equal(proof[:, lo:hi], po[:, lo:hi]) and np.array_equal(status[lo:hi], so[lo:hi])
    assert (proof[:, :lo] == 0).all() and (status[:lo] == 0xEE).all() and (status[hi:] == 0xEE).all()
    # device: same with torch views
    dev = torch.device("cuda", 0)
    w, r, c = (torch.from_numpy(x).to(dev) for x in (wo, ro, co))
    pd = torch.zeros((27, N), dtype=torch.uint8, device=dev); sd = torch.full((N,), 0xEE, dtype=torch.uint8, device=dev)
    ctx.prove_batch(w[:, lo:hi], r[:, lo:hi], c[:, lo:hi], proof=pd[:, lo:hi], status=sd[lo:hi])
    ctx.sync()
    assert np.array_equal(pd.cpu().numpy(), proof) and np.array_equal(sd.cpu().numpy(), status)
    # empty batches are a no-op
    p0, s0 = ctx.prove_batch(np.zeros((12, 0), np.uint8), np.zeros((9, 0), np.uint8), np.zeros((5, 0), np.uint8))
    assert p0.shape == (27, 0) and s0.shape == (0,)
    assert ctx.verify_batch(np.zeros((27, 0), np.uint8), np.zeros((5, 0), np.uint8), np.zeros((0,), np.uint8)).shape == (0,)


@pytest.mark.parametrize("n", (1, 255, 256, 257, 30037, 65536 + 19))
def test_tma_tiles_ragged_and_aligned(gpu_ctx, oracle, n):
    """The TMA path needs 16-byte aligned bases and pitches; ragged item counts ride on an aligned pitch and the hardware
    clips the last tile.  Same bytes as the plain-load path and the oracle, and nothing is written past item n."""
    import torch
    ctx = gpu_ctx["table"]
    pitch = (n + 64 + 15) // 16 * 16
    dev = torch.device("cuda", 0)
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=n, dist=0)
    po, so = oracle.prove_batch(wo, ro, co)
    big = lambda planes: torch.full((planes, pitch), 0xAB, dtype=torch.uint8, device=dev)
    W, R, Cc, P = big(12), big(9), big(5), big(27)
    W[:, :n] = torch.from_numpy(wo).to(dev); R[:, :n] = torch.from_numpy(ro).to(dev); Cc[:, :n] = torch.from_numpy(co).to(dev)
    S = torch.full((pitch,), 0xAB, dtype=torch.uint8, device=dev)
    ctx.prove_batch(W[:, :n], R[:, :n], Cc[:, :n], proof=P[:, :n], status=S[:n])
    ctx.sync()
    assert np.array_equal(P[:, :n].cpu().numpy(), po) and np.array_equal(S[:n].cpu().numpy(), so)
    assert bool((P[:, n:] == 0xAB).all()) and bool((S[n:] == 0xAB).all())


@pytest.mark.parametrize("chunk_log2", (8, 12, 17))
def test_host_pipeline_chunks_and_fused_call(product_lib, oracle, chunk_log2):
    """Host-pointer entry points with several chunk sizes (many chunks cycling through the staging slots), and the fused
    prove+verify extension: same bytes as the two separate calls and as the oracle."""
    import pbh_b200
    n = 70000 + 3
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=chunk_log2, dist=0, threads=8)
    po, so = oracle.prove_batch(wo, ro, co, threads=8)
    vo = oracle.verify_batch(po, co, uo, threads=8, want_gt=False)
    with pbh_b200.Context(device=0) as ctx:
        ctx.set_option(pbh_b200.OPT_CHUNK_LOG2, chunk_log2)
        p, s = ctx.prove_batch(wo, ro, co)
        v = ctx.verify_batch(po, co, uo)
        assert np.array_equal(p, po) and np.array_equal(s, so) and np.array_equal(v, vo)
        p2, s2, v2 = ctx.prove_verify_batch(wo, ro, co, uo)
        assert np.array_equal(p2, po) and np.array_equal(s2, so) and np.array_equal(v2, vo)


@pytest.mark.parametrize("n,pitch", ((1, 16), (255, 256), (4099, 4099), (70003, 70016), (70003, 70004)))
def test_pinned_host_buffers_run_in_place(product_lib, oracle, n, pitch):
    """Page-locked, mapped host buffers: the kernels run in place on them (PBH_OPT_HOST_DIRECT), TMA tiles when base and
    pitch are 16-byte aligned, plain loads/stores otherwise.  Same bytes as the staged path and as the oracle; bytes
    beyond the n items of each plane are never written; the verifier's GT output takes the same path."""
    import torch
    import pbh_b200
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=pitch, dist=0, threads=8)
    po, so = oracle.prove_batch(wo, ro, co, threads=8)
    vo, go = oracle.verify_batch(po, co, uo, threads=8, want_gt=True)

    def pinned(planes, src=None):
        t = torch.full((planes, pitch), 0xAB, dtype=torch.uint8).pin_memory()
        if src is not None:
            t[:, :n] = torch.from_numpy(np.atleast_2d(src))
        return t

    W, R, Cc, U = pinned(12, wo), pinned(9, ro), pinned(5, co), pinned(1, uo)
    with pbh_b200.Context(device=0) as ctx:
        launches = {}
        for direct in (1, 0):
            ctx.set_option(pbh_b200.OPT_HOST_DIRECT, direct)
            P, S, V, G = pinned(27), pinned(1), pinned(1), pinned(4)
            l0 = ctx.launch_count
            ctx.prove_batch(W.numpy()[:, :n], R.numpy()[:, :n], Cc.numpy()[:, :n], proof=P.numpy()[:, :n], status=S.numpy()[0, :n])
            ctx.verify_batch(P.numpy()[:, :n], Cc.numpy()[:, :n], U.numpy()[0, :n], result=V.numpy()[0, :n], gt=G.numpy()[:, :n])
            launches[direct] = ctx.launch_count - l0
            assert np.array_equal(P.numpy()[:, :n], po) and np.array_equal(S.numpy()[0, :n], so)
            assert np.array_equal(V.numpy()[0, :n], vo) and np.array_equal(G.numpy()[:, :n], go)
            for t in (P, S, V, G):
                assert bool((t[:, n:] == 0xAB).all())
        assert launches[1] == 2      # one prover launch, one verifier launch: no chunking on the in-place path


_FUSED_CACHE = {}


def _fused_case(n, first):
    if n not in _FUSED_CACHE:
        import oracle as O
        wo, ro, co, uo, _ = O.generate_inputs(n, first_index=first, seed=9, dist=1 if n > 100 else 0, threads=8)
        po, so = O.prove_batch(wo, ro, co, threads=8)
        vo = O.verify_batch(po, co, uo, threads=8, want_gt=False)
        _FUSED_CACHE[n] = (wo, ro, co, uo, po, so, vo)
    return _FUSED_CACHE[n]


@pytest.mark.parametrize("algo", CTXS)
@pytest.mark.parametrize("n", (5, 1000, 65536 + 77))
def test_fused_digest_and_bitmap(gpu_ctx, oracle, algo, n):
    """pbh_prove_digest_batch_dev / pbh_verify_bitmap_batch_dev == plain calls + pbh_digest_dev / pbh_pack_verdicts_dev == oracle,
    on the TMA path (aligned pitch) and on the fallback paths."""
    import torch
    ctx = gpu_ctx[algo]
    dev = torch.device("cuda", 0)
    first = 12345678901
    wo, ro, co, uo, po, so, vo = _fused_case(n, first)
    for pitch in (n, (n + 15) // 16 * 16):
        mk = lambda planes, src: (lambda t: (t[:, :n].copy_(torch.from_numpy(src).to(dev)), t[:, :n])[1])(
            torch.zeros((planes, pitch), dtype=torch.uint8, device=dev))
        w, r, c = mk(12, wo), mk(9, ro), mk(5, co)
        u = torch.from_numpy(uo).to(dev)
        proof = torch.zeros((27, pitch), dtype=torch.uint8, device=dev)[:, :n]
        status = torch.zeros((n,), dtype=torch.uint8, device=dev); result = torch.zeros((n,), dtype=torch.uint8, device=dev)
        digest = torch.zeros((1,), dtype=torch.int64, device=dev)
        bitmap = torch.full(((n + 7) // 8 + 8,), 0xEE, dtype=torch.uint8, device=dev)
        ctx.prove_digest_batch(w, r, c, proof, status, digest, first_index=first)
        ctx.verify_bitmap_batch(proof, c, u, result, bitmap[: (n + 7) // 8])
        ctx.sync()
        assert np.array_equal(proof.cpu().numpy(), po) and np.array_equal(status.cpu().numpy(), so)
        assert np.array_equal(result.cpu().numpy(), vo)
        assert (int(digest.item()) & (2**64 - 1)) == oracle.digest(po, first_index=first)
        assert np.array_equal(bitmap[: (n + 7) // 8].cpu().numpy(), oracle.pack_verdicts(vo))
        assert bool((bitmap[(n + 7) // 8:] == 0xEE).all())


def test_shard_summaries(gpu_ctx, oracle):
    """Verdict bitmaps and additive digests: identical whatever the shard count (SURVEY.md §8e)."""
    import torch
    ctx = gpu_ctx["table"]
    n = 100003
    w, r, c, u = ctx.generate_inputs(n, seed=5, dist=1)
    proof, status = ctx.prove_batch(w, r, c)
    res = ctx.verify_batch(proof, c, u)
    bits = ctx.pack_verdicts(res)
    dig = ctx.digest(proof)
    ctx.sync()
    assert np.array_equal(bits.cpu().numpy(), oracle.pack_verdicts(res.cpu().numpy()))
    whole = int(dig.item()) & (2**64 - 1)
    assert whole == oracle.digest(proof.cpu().numpy())
    for shards in (2, 4, 8):
        total = 0
        parts = []
        for g in range(shards):
            lo, hi = g * n // shards, (g + 1) * n // shards
            wg, rg, cg, ug = ctx.generate_inputs(hi - lo, first_index=lo, seed=5, dist=1)
            pg, sg = ctx.prove_batch(wg, rg, cg)
            vg = ctx.verify_batch(pg, cg, ug)
            total = (total + (int(ctx.digest(pg, first_index=lo).item()) & (2**64 - 1))) % 2**64
            parts.append(vg)
        ctx.sync()
        assert total == whole
        assert torch.equal(torch.cat(parts), res)


# ---------------------------------------------------------------------------------------------
# BASELINE.json sizes: size-independent properties (the oracle is too slow to replay 2^20+ items here)
# ---------------------------------------------------------------------------------------------
def test_full_size_properties(gpu_ctx, oracle):
    import torch
    n = 1 << 20
    t, a = gpu_ctx["table"], gpu_ctx["arith"]
    w, r, c, u = t.generate_inputs(n, seed=0xB200, dist=1)
    pt, st = t.prove_batch(w, r, c)
    pa, sa = a.prove_batch(w, r, c)
    pi, si = gpu_ctx["table_int"].prove_batch(w, r, c)
    gpu_ctx["table_int"].sync()
    assert torch.equal(pt, pi) and torch.equal(st, si)
    vt, gt_t = t.verify_batch(pt, c, u, want_gt=True)
    va, gt_a = a.verify_batch(pa, c, u, want_gt=True)
    t.sync(); a.sync()
    # (1) D_fullpath: every item proves and reaches the pairing check; (2) the two algorithms agree byte for byte;
    assert int((st != 0).sum()) == 0 and torch.equal(pt, pa) and torch.equal(st, sa)
    assert torch.equal(vt, va) and torch.equal(gt_t, gt_a)
    assert int(((vt != 0) & (vt != 1)).sum()) == 0
    # (3) accept <=> e1 == e2
    eq = (gt_t[0] == gt_t[2]) & (gt_t[1] == gt_t[3])
    assert torch.equal(eq, vt == 1)
    # (4) an oracle-checked prefix and a strided sample
    idx = torch.arange(0, n, 997, device=w.device)
    wo, ro, co, uo = (x[..., idx].cpu().numpy() for x in (w, r, c, u))
    po, so = oracle.prove_batch(wo, ro, co, threads=8)
    vo, go = oracle.verify_batch(po, co, uo, threads=8)
    assert np.array_equal(pt[:, idx].cpu().numpy(), po) and np.array_equal(vt[idx].cpu().numpy(), vo)
    assert np.array_equal(gt_t[:, idx].cpu().numpy(), go)
    # (5) tampering one evaluation of an accepted proof never yields a different accepted GT pair silently: verdicts of
    #     a tampered batch agree between the algorithms
    p2 = pt.clone(); p2[25] = (p2[25] + 1) % 17
    assert torch.equal(t.verify_batch(p2, c, u), a.verify_batch(p2, c, u))
    # (6) uniform inputs at full size: the status histogram matches SURVEY.md §2.4 within sampling error
    wu, ru, cu, uu = t.generate_inputs(n, seed=1, dist=0)
    pu, su = t.prove_batch(wu, ru, cu)
    vu = t.verify_batch(pu, cu, uu)
    pui, sui = gpu_ctx["table_int"].prove_batch(wu, ru, cu)
    t.sync(); gpu_ctx["table_int"].sync()
    assert torch.equal(pu, pui) and torch.equal(su, sui)      # FP32-pipe prover == int32 prover on 2^20 uniform items
    hist = torch.bincount(su.to(torch.int64), minlength=6).cpu().numpy() / n
    assert abs(hist[2] - 0.424) < 0.01 and abs(hist[4] - 0.149) < 0.01 and abs(hist[5] - 0.315) < 0.01 and hist[3] < 0.002
    ok = su == 0
    acc = float(((vu == 1) & ok).sum()) / n
    assert abs(acc - 0.032) < 0.005


def test_config2_verifier_16m(gpu_ctx, oracle):
    """BASELINE.json configs[2]: 16 M proofs through the verifier.  Size-independent properties: the two verifier
    algorithms (group tables vs per-item curve arithmetic + Miller loop) agree byte for byte, accept <=> e1 == e2,
    tampered evaluations never raise the acceptance count, an oracle-checked strided sample."""
    import torch
    n = 1 << 24
    t, a = gpu_ctx["table"], gpu_ctx["arith"]
    w, r, c, u = t.generate_inputs(n, seed=0xB200, dist=1)
    proof, status = t.prove_batch(w, r, c)
    vt, gt_t = t.verify_batch(proof, c, u, want_gt=True)
    va, gt_a = a.verify_batch(proof, c, u, want_gt=True)
    t.sync(); a.sync()
    assert int((status != 0).sum()) == 0
    assert torch.equal(vt, va) and torch.equal(gt_t, gt_a)
    assert torch.equal((gt_t[0] == gt_t[2]) & (gt_t[1] == gt_t[3]), vt == 1)
    accepted = int((vt == 1).sum())
    assert 0.55 < accepted / n < 0.75                     # ~63 % of full-path items verify (SURVEY.md §2.4: 3.2 / 5.1)
    bad = proof.clone(); bad[20] = (bad[20] + 1) % 17      # a_z tampered everywhere
    vb = t.verify_batch(bad, c, u)
    t.sync()
    assert int(((vb != 0) & (vb != 1)).sum()) == 0 and int((vb == 1).sum()) < accepted
    idx = torch.arange(0, n, 40009, device=w.device)
    po, so = oracle.prove_batch(*(x[..., idx].cpu().numpy() for x in (w, r, c)), threads=8)
    vo, go = oracle.verify_batch(po, c[:, idx].cpu().numpy(), u[idx].cpu().numpy(), threads=8)
    assert np.array_equal(proof[:, idx].cpu().numpy(), po) and np.array_equal(vt[idx].cpu().numpy(), vo)
    assert np.array_equal(gt_t[:, idx].cpu().numpy(), go)


def test_config4_256m_end_to_end_sharding(gpu_ctx, oracle):
    """BASELINE.json configs[4] at full size on one GPU: 2^28 witnesses proved and verified as 1 shard and as 8 shards
    (the ranks of an 8-GPU run, executed one after the other here): identical verdict bitmaps, digests add up."""
    import torch
    from pbh_b200 import sharding
    ctx = gpu_ctx["table"]
    n = 1 << 28
    dev = torch.device("cuda", 0)

    def run(first, count):
        w, r, c, u = ctx.generate_inputs(count, first_index=first, seed=0xB200, dist=1)
        proof = torch.empty((27, count), dtype=torch.uint8, device=dev); status = torch.empty((count,), dtype=torch.uint8, device=dev)
        result = torch.empty((count,), dtype=torch.uint8, device=dev); bitmap = torch.empty((count // 8,), dtype=torch.uint8, device=dev)
        digest = torch.empty((1,), dtype=torch.int64, device=dev)
        ctx.prove_digest_batch(w, r, c, proof, status, digest, first_index=first)
        ctx.verify_bitmap_batch(proof, c, u, result, bitmap)
        ctx.sync()
        ok = int((status != 0).sum()) == 0
        sample = (proof[:, ::(1 << 20) + 7].cpu().numpy(), w[:, ::(1 << 20) + 7].cpu().numpy(), r[:, ::(1 << 20) + 7].cpu().numpy(),
                  c[:, ::(1 << 20) + 7].cpu().numpy())
        return bitmap, int(digest.item()) & (2**64 - 1), ok, sample

    whole_bitmap, whole_digest, ok, sample = run(0, n)
    assert ok
    po, so = oracle.prove_batch(sample[1], sample[2], sample[3], threads=8)
    assert np.array_equal(sample[0], po)                    # an oracle-checked strided sample of the 2^28 proofs
    whole_bitmap = whole_bitmap.cpu()
    total = 0
    parts = []
    for rank in range(8):
        lo, hi = sharding.shard_range(n, rank, 8)
        b, d, ok, _ = run(lo, hi - lo)
        assert ok
        parts.append(b.cpu()); total = (total + d) % 2**64
    assert total == whole_digest
    assert torch.equal(torch.cat(parts), whole_bitmap)


@pytest.mark.parametrize("algo", ("table", "arith"))
def test_record_wire_format(gpu_ctx, oracle, algo):
    """SURVEY.md §8(f) row 3: 32-byte array-of-structs records in, records out — same bytes as the plane API and the oracle."""
    import pbh_b200
    ctx = gpu_ctx[algo]
    n = 300000 + 11                      # more than one staged chunk
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=41, dist=0, threads=8)
    po, so = oracle.prove_batch(wo, ro, co, threads=8)
    vo = oracle.verify_batch(po, co, uo, threads=8, want_gt=False)
    assert pbh_b200.WITNESS_RECORD.itemsize == 32 and pbh_b200.PROOF_RECORD.itemsize == 32
    wrec = pbh_b200.witness_records(wo, ro, co, uo)
    wrec["reserved"] = 0xAA              # ignored on input
    prec = ctx.prove_records(wrec)
    p, s = pbh_b200.proof_planes(prec)
    assert np.array_equal(p, po) and np.array_equal(s, so) and not prec["reserved"].any()
    res = ctx.verify_records(pbh_b200.proof_records(po, so), wrec)
    assert np.array_equal(res, vo)
    assert ctx.prove_records(wrec[:0]).shape == (0,)


@pytest.mark.parametrize("algo", ("table", "arith"))
def test_fuzz_arbitrary_bytes(gpu_ctx, oracle, algo):
    """Every input byte may take any of the 256 values (2 % of bytes are replaced by uniform random bytes): the status /
    result classes, the zeroed outputs and every other byte still match the oracle; nothing is read or written out of
    bounds (the verdict of a malformed item is decided before any table is indexed)."""
    ctx = gpu_ctx[algo]
    rng = np.random.default_rng(123)
    n = 120000
    wo, ro, co, uo, _ = oracle.generate_inputs(n, seed=55, dist=1, threads=8)
    po, _ = oracle.prove_batch(wo, ro, co, threads=8)

    def corrupt(a):
        a = a.copy()
        mask = rng.random(a.shape) < 0.02
        a[mask] = rng.integers(0, 256, size=int(mask.sum()), dtype=np.uint8)
        return a

    w2, r2, c2 = corrupt(wo), corrupt(ro), corrupt(co)
    pe, se = oracle.prove_batch(w2, r2, c2, threads=8)
    p, s = ctx.prove_batch(w2, r2, c2)
    assert np.array_equal(s, se) and np.array_equal(p, pe)
    assert (se == 32).sum() > 0 and (se == 0).sum() > 0
    p3, c3, u3 = corrupt(po), corrupt(co), corrupt(uo)
    ve, ge = oracle.verify_batch(p3, c3, u3, threads=8)
    v, g = ctx.verify_batch(p3, c3, u3, want_gt=True)
    assert np.array_equal(v, ve) and np.array_equal(g, ge)
    assert set(np.unique(ve)) >= {0, 1, 2, 4, 0x20}
