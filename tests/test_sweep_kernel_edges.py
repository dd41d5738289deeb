"""The input generator, the generic NTT and NTT product, the polynomial product, the KZG commitment across SRSs, the general
division, the ragged add / subtract and the record transposes, at the path and context edges no other test reaches.

Every device call works on planes placed at chosen offsets and pitches inside guard-filled buffers (0xA5, or 0xA5A5 for the
uint16 planes of the NTTs): outputs are compared with an exact reference, every byte outside them must keep its guard value,
and inputs must come back untouched.  Grids are capped at SM count x 8 x 256 threads (grid_for(ctx, ., 8) of each entry
point), so one case per kernel runs past the cap and ends in a ragged part.  The first call of each case also runs under
torch.profiler and must launch exactly the kernels the dispatch in pbh_capi.cu names.

Two defects these tests pinned down:
  - PBH_DIST_FULLPATH searched attempts without bound, so a context whose circuit no witness of the generator's table
    satisfies (or whose SRS is too short for any proof) never returned.  The search now stops at PBH_GEN_MAX_ATTEMPTS in
    the kernel and the oracle, and the first case is refused on the host with PBH_ERR_UNSUPPORTED before any launch.
  - pbh_ntt_generic_batch refused FORWARD transforms whose length has no inverse modulo the modulus (modulus 2, even
    moduli), which the reference computes: only fft_inv needs the inverse.
"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from test_kernel_instantiations import SWEEP_KERNELS, _profiled_kernels

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 0xA5
PER_SM = 8                                     # grid_for(ctx, ., 8) of every entry point here
BLOCK = 256
OK, BAD_ARGUMENT, SETUP_PANIC, UNSUPPORTED = 0, -1, -2, -5


def gen_max_attempts():
    with open(os.path.join(ROOT, "include", "pbh_b200.h")) as f:
        return int(re.search(r"#define PBH_GEN_MAX_ATTEMPTS (\d+)", f.read()).group(1))


# ---------------------------------------------------------------------------------------------
# placement: planes at an offset and pitch (in elements) inside a guard-filled buffer
# ---------------------------------------------------------------------------------------------
class Buf:
    """`planes` planes of `n` elements, `pitch` elements apart, from element `off` of a guard-filled buffer (a CUDA byte
    tensor when `dev`, else numpy).  `x` (planes, n) is written in; outputs pass x=None with planes and n."""

    def __init__(self, x, off, pitch, dev, dtype=np.uint8, planes=None, n=None):
        self.dtype, self.dev, self.off, self.pitch = np.dtype(dtype), dev, off, pitch
        self.planes, self.n = (x.shape if x is not None else (planes, n))
        assert pitch >= self.n
        g = GUARD if self.dtype.itemsize == 1 else GUARD * 0x0101
        self.host = np.full(off + self.planes * pitch + 64, g, self.dtype)
        self.guard_image = self.host.copy()
        if x is not None:
            self.view(self.host)[...] = x
        self.image = self.host.copy()
        if dev:
            import torch
            self.t = torch.from_numpy(self.host.view(np.uint8)).cuda()
            assert self.t.data_ptr() % 256 == 0
            self.ptr = self.t.data_ptr() + off * self.dtype.itemsize
        else:
            self.ptr = self.host.ctypes.data + off * self.dtype.itemsize

    def view(self, arr):
        s = self.dtype.itemsize
        return np.lib.stride_tricks.as_strided(arr[self.off:], shape=(self.planes, self.n), strides=(self.pitch * s, s))

    def fetch(self):
        return self.t.cpu().numpy().view(self.dtype) if self.dev else self.host.copy()

    def check(self, want, what):
        """Output: the planes equal `want`, every other element still holds the guard."""
        h = self.fetch()
        got = self.view(h).copy()
        if not np.array_equal(got, want):
            bad = np.argwhere(got != want)
            raise AssertionError(f"{what}: {len(bad)} elements differ, first (plane, item) {tuple(bad[0])}: got {got[tuple(bad[0])]}, "
                                 f"want {want[tuple(bad[0])]}")
        self.view(h)[...] = self.view(self.guard_image)
        assert np.array_equal(h, self.guard_image), f"{what}: guard elements overwritten"

    def untouched(self, what):
        assert np.array_equal(self.fetch(), self.image), f"{what}: input modified"

    def settle(self):
        """An output that becomes the next call's input: its current contents are the snapshot `untouched` compares."""
        self.image = self.fetch()


def _pp(b):
    return C.c_void_p(b.ptr), C.c_size_t(b.pitch)


def _null_pp():
    return C.c_void_p(None), C.c_size_t(0)


def grid_cap():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * PER_SM * BLOCK


def place(role, slot, n, aligned=True):
    """(offset, pitch) in elements: aligned placements keep every base and pitch a multiple of 16 elements' worth of 4 bytes;
    the others put bases and pitches on odd elements.  Every buffer gets its own pitch."""
    room = -(-n // 16) * 16 + 16 * (slot + 1) + (32 if role == "out" else 0)
    return (16 * (slot + 1), room) if aligned else (2 * slot + 1, room + 2 * slot + 1)


def _families():
    return {re.match(r"\w+", k).group(0) for k in SWEEP_KERNELS}


CENSUS = {}


def census(key, fn):
    """Runs `fn` once; the first time per `key` under the profiler, returning the product kernels it launched (None when
    the profiler records no kernels on this machine, or the key was seen)."""
    if key in CENSUS:
        fn()
        return None
    fams = _families()
    names = [k for k in _profiled_kernels(fn) if re.match(r"\w+", k).group(0) in fams]
    CENSUS[key] = names
    return names


def assert_census(key, fn, want):
    names = census(key, fn)
    if names is not None and CENSUS.get("_profiler_works", True):
        assert names == want, (key, names, want)


@pytest.fixture(scope="module")
def profiler_ok():
    import torch
    x = torch.arange(1 << 16, device="cuda", dtype=torch.float32)
    ok = len(_profiled_kernels(lambda: x.mul_(2.0))) > 0
    CENSUS["_profiler_works"] = ok
    return ok


# =============================================================================================
# 1. the input generator
# =============================================================================================
def reference_circuit(mod):
    return mod.pbh_test_circuit()


def unsatisfiable_circuit(mod):
    c = mod.pbh_test_circuit()
    c.q_c[3] = 2                   # the add gate becomes a + b - c + 2 = 0: no row (x, y, z, x^2 ...) of the table satisfies it
    return c


def scaled_circuit(mod):
    """Every gate's five selectors times a different non-zero constant: the same solutions, other selector polynomials."""
    c = mod.pbh_test_circuit()
    for g, k in enumerate((3, 5, 16, 7)):
        for name in ("q_l", "q_r", "q_o", "q_m", "q_c"):
            getattr(c, name)[g] = getattr(c, name)[g] * k % 17
    return c


def split_circuit(mod):
    """Every copy cycle of the reference circuit is a transposition, so running a cycle the other way changes nothing.
    Instead the cycle c[2] <-> c[3] is split into two fixed points: fewer equalities, which the table still satisfies,
    and other sigma polynomials."""
    c = mod.pbh_test_circuit()
    wires = [list(c.c_a_wire), list(c.c_b_wire), list(c.c_c_wire)]
    idxs = [list(c.c_a_index), list(c.c_b_index), list(c.c_c_index)]
    perm = {(w, i): (wires[w][i], idxs[w][i] - 1) for w in range(3) for i in range(4)}
    assert all(perm[perm[p]] == p for p in perm) and perm[(2, 2)] == (2, 3)
    c.c_c_wire[2] = c.c_c_wire[3] = 2
    c.c_c_index[2], c.c_c_index[3] = 3, 4
    return c


CIRCUITS = {"reference": reference_circuit, "scaled": scaled_circuit, "split": split_circuit}
GEN_CONTEXTS = [("reference", 2, 6), ("reference", 3, 6), ("reference", 5, 7), ("reference", 2, 9), ("scaled", 2, 6),
                ("split", 3, 6)]
FIRST_INDICES = (0, 2**32 - 5, 2**40 + 3)
SHORT_SRS = (2, 5)             # every full-path attempt fails on this SRS: the attempt cap decides


def _oracle_gen(oracle, n, first, seed, dist, circ, s, srs_n):
    return oracle.generate_inputs(n, first_index=first, seed=seed, dist=dist, circuit=circ, s=s, srs_n=srs_n,
                                  threads=oracle.hardware_threads() or 4)


_BOUNDED = r"""
import sys, numpy as np
sys.path.insert(0, {oracle!r})
import oracle as O
c = O.pbh_test_circuit()
if {unsat}:
    c.q_c[3] = 2
w0, r0, c0, u0, _ = O.generate_inputs(24, first_index=7, seed=11, dist=0, circuit=c, s={s}, srs_n={srs_n}, threads=8)
w1, r1, c1, u1, a1 = O.generate_inputs(24, first_index=7, seed=11, dist=1, circuit=c, s={s}, srs_n={srs_n}, threads=8)
assert (a1 == 255).all(), a1
for x, y in ((w0, w1), (r0, r1), (c0, c1), (u0, u1)):
    assert np.array_equal(x, y)
print("bounded")
"""


@pytest.mark.parametrize("case", ["unsatisfiable", "short_srs"])
def test_oracle_fullpath_search_is_bounded(oracle, case):
    """The oracle's full-path search ends after PBH_GEN_MAX_ATTEMPTS attempts with attempt 0's draw and attempt byte 255,
    on a circuit no table row satisfies and on an SRS too short for any proof.  In a subprocess, so that an unbounded
    search fails the test instead of hanging the suite."""
    s, srs_n = (2, 6) if case == "unsatisfiable" else SHORT_SRS
    code = _BOUNDED.format(oracle=os.path.join(ROOT, "oracle"), unsat=case == "unsatisfiable", s=s, srs_n=srs_n)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and "bounded" in r.stdout, r.stderr[-2000:]


def test_oracle_fullpath_unchanged_below_the_cap(oracle):
    """On the reference circuit the cap is far out of reach: every item of a 2^16 batch succeeds, at attempts the
    geometric law of a ~1/19 success rate predicts."""
    *_, att = _oracle_gen(oracle, 1 << 16, 0, 0xB200, 1, oracle.pbh_test_circuit(), 2, 6)
    assert att.max() < 255 and 10 < att.mean() < 30
    assert gen_max_attempts() == 4096


def test_generator_circuits_satisfiable_by_the_table():
    """The scaled and rotated circuits keep the reference's solutions; the unsatisfiable one has none in the table."""
    import oracle as O
    rows = [(x, y, z) for x in range(17) for y in range(17) for z in range(17) if (x * x + y * y - z * z) % 17 == 0]
    assert len(rows) == 289

    def sat(c, x, y, z):
        w = [x, y, z, x * x % 17, x, y, z, y * y % 17, x * x % 17, y * y % 17, z * z % 17, z * z % 17]
        a, b, cc = w[:4], w[4:8], w[8:]
        for g in range(4):                      # Q8: q_l where q_r is meant
            if (c.q_l[g] * a[g] + c.q_l[g] * b[g] + c.q_o[g] * cc[g] + c.q_m[g] * a[g] * b[g] + c.q_c[g]) % 17:
                return False
        wires = (a, b, cc)
        for wv, (ws, ix) in enumerate(((c.c_a_wire, c.c_a_index), (c.c_b_wire, c.c_b_index), (c.c_c_wire, c.c_c_index))):
            if any(wires[wv][g] != wires[ws[g]][ix[g] - 1] for g in range(4)):
                return False
        return True

    for name, make in CIRCUITS.items():
        assert sum(sat(make(O), *r) for r in rows) > 0, name
    assert sum(sat(unsatisfiable_circuit(O), *r) for r in rows) == 0


def _gen_call(ctx, n, first, seed, dist, placed, attempt):
    return ctx.lib.pbh_generate_inputs_dev(ctx.h, C.c_size_t(n), C.c_uint64(first), C.c_uint64(seed), int(dist),
                                           *_pp(placed[0]), *_pp(placed[1]), *_pp(placed[2]), C.c_void_p(placed[3].ptr),
                                           C.c_void_p(attempt.ptr if attempt is not None else None))


def run_generate(ctx, oracle, n, first, seed, dist, circ, s, srs_n, with_attempt=True, aligned=True, key=None):
    outs = [Buf(None, *place("out", k, n, aligned), True, planes=p, n=n) for k, p in enumerate((12, 9, 5, 1))]
    att = Buf(None, *place("out", 4, n, aligned), True, planes=1, n=n) if with_attempt else None
    fn = lambda: ctx._check(_gen_call(ctx, n, first, seed, dist, outs, att), "pbh_generate_inputs_dev") or ctx.sync()
    if key:
        assert_census(key, fn, ["generate_kernel"])
    else:
        fn()
    want = _oracle_gen(oracle, n, first, seed, dist, circ, s, srs_n)
    for b, w, name in zip(outs, want[:3] + (want[3][None],), ("wit", "rand", "chal", "u")):
        b.check(w, f"generate {name} n={n} first={first} dist={dist} srs=({s},{srs_n})")
    if att is not None:
        att.check(want[4][None], f"generate attempt n={n} first={first}")
    return want


@gpu
@pytest.mark.parametrize("ctx_case", GEN_CONTEXTS, ids=[f"{c}-s{s}-n{n}" for c, s, n in GEN_CONTEXTS])
def test_generator_matches_the_oracle(oracle, profiler_ok, ctx_case):
    """wit / rand / chal / u / attempt byte for byte, both distributions, three first indices (two beyond 32 bits), pitches
    > n inside guard bytes, with and without the attempt plane."""
    import pbh_b200 as P
    name, s, srs_n = ctx_case
    with P.Context(circuit=CIRCUITS[name](P), s=s, srs_n=srs_n, device=0) as ctx:
        circ = CIRCUITS[name](oracle)
        for dist in (0, 1):
            for first in FIRST_INDICES:
                want = run_generate(ctx, oracle, 1031, first, 0x5EED + s, dist, circ, s, srs_n, with_attempt=first != 2**32 - 5,
                                    aligned=first != 0, key=("generate", name, s, srs_n, dist, first) if first == 0 else None)
                if first:                            # not the items whose index is the global index truncated to 32 bits
                    idx = (first + np.arange(1031)) % 2**32
                    near = idx < 2048
                    alias = _oracle_gen(oracle, 2048, 0, 0x5EED + s, dist, circ, s, srs_n)
                    assert near.sum() > 1000
                    assert not np.array_equal(alias[0][:, idx[near]], want[0][:, near])
                    assert not np.array_equal(alias[1][:, idx[near]], want[1][:, near])
            if dist == 1:
                assert want[4].max() < 255


@gpu
def test_generator_past_the_grid_cap(oracle):
    """More items than the capped grid has threads, ending in a ragged part, on both distributions."""
    import pbh_b200 as P
    n = grid_cap() + BLOCK // 2 + 3
    with P.Context(device=0) as ctx:
        for dist in (0, 1):
            run_generate(ctx, oracle, n, 2**40 + 3, 0xCAFE, dist, oracle.pbh_test_circuit(), 2, 6)


@gpu
def test_generator_attempt_cap_on_a_short_srs(oracle):
    """SRS(2, 5): every full-path attempt fails, so the kernel stops at PBH_GEN_MAX_ATTEMPTS like the oracle: attempt 0's
    draw, attempt byte 255."""
    import pbh_b200 as P
    s, srs_n = SHORT_SRS
    with P.Context(s=s, srs_n=srs_n, device=0) as ctx:
        want = run_generate(ctx, oracle, 301, 2**32 - 5, 7, 1, oracle.pbh_test_circuit(), s, srs_n)
        assert (want[4] == 255).all()
        uni = _oracle_gen(oracle, 301, 2**32 - 5, 7, 0, oracle.pbh_test_circuit(), s, srs_n)
        assert all(np.array_equal(a, b) for a, b in zip(want[:4], uni[:4]))


@gpu
def test_generator_refuses_an_unsatisfiable_circuit(oracle):
    """No table row satisfies the circuit: PBH_DIST_FULLPATH is refused on the host, before any launch, through the
    context and through the sharded multi-device pass; the uniform distribution still generates."""
    import pbh_b200 as P
    with P.Context(circuit=unsatisfiable_circuit(P), device=0) as ctx:
        before = ctx.launch_count
        with pytest.raises(P.PbhError, match="PBH_ERR_UNSUPPORTED"):
            ctx.generate_inputs(1000, dist=P.DIST_FULLPATH)
        assert ctx.launch_count == before
        run_generate(ctx, oracle, 1000, 5, 9, 0, unsatisfiable_circuit(oracle), 2, 6)
    with P.MultiContext([0], circuit=unsatisfiable_circuit(P)) as m:
        for fn in (m.prove_verify_sharded, m.prove_verify_fs_sharded):
            with pytest.raises(P.PbhError, match="UNSUPPORTED"):
                fn(4096, dist=P.DIST_FULLPATH)


# =============================================================================================
# 2. generic NTT and NTT product
# =============================================================================================
def _ct(vals, dom, m):
    """The reference's recursive Cooley-Tukey (src/fft.rs:81-106) on lists of numpy item vectors."""
    if len(vals) == 1:
        return [vals[0]]
    half = dom[0::2]
    l, r = _ct(vals[0::2], half, m), _ct(vals[1::2], half, m)
    o = [None] * len(vals)
    for i in range(min(len(l), len(r))):
        y = r[i] * dom[i] % m
        o[i] = (l[i] + y) % m
        o[i + len(vals) // 2] = (l[i] - y) % m
    return o


def ref_fft(x, m, omega, inverse=False):
    """CooleyTurkey::fft / fft_inv (src/fft.rs:51-79) over Z_m, exact, on (size, n) arrays; values reduced first as F::from
    reduces them.  ArithmeticError where fft_inv's `F::from(len).inv().unwrap()` panics."""
    size = x.shape[0]
    dom, p = [], 1 % m
    for _ in range(size):
        dom.append(p)
        p = p * (omega % m) % m
    out = _ct([np.asarray(v, dtype=np.int64) % m for v in x], dom, m)
    if inverse:
        try:
            inv = pow(size, -1, m)
        except ValueError:
            raise ArithmeticError("fft_inv: len has no inverse")
        out = [out[0] * inv % m] + [out[size - k] * inv % m for k in range(1, size)]
    return np.stack(out).astype(np.uint16)


def ref_mul_ntt(a, b, m, omega):
    """mul_ntt (src/fft.rs:109-132): both zero-extended to la + lb, transformed, multiplied pointwise, fft_inv."""
    size = a.shape[0] + b.shape[0]
    za = np.zeros((size, a.shape[1]), np.int64); za[:a.shape[0]] = a
    zb = np.zeros((size, b.shape[1]), np.int64); zb[:b.shape[0]] = b
    fa, fb = ref_fft(za, m, omega).astype(np.int64), ref_fft(zb, m, omega).astype(np.int64)
    return ref_fft(fa * fb % m, m, omega, inverse=True)


def _primitive(m, size):
    """An element of order exactly `size` modulo the prime m, or None."""
    if (m - 1) % size:
        return None
    for g in range(2, m):
        w = pow(g, (m - 1) // size, m)
        if pow(w, size // 2, m) != 1:
            return w
    return None


SIZES = (2, 4, 8, 16, 32, 64)
MODULI = (2, 3, 5, 17, 97, 257, 337, 7681, 12289, 40961, 65521, 12)    # 12: an even composite


def omegas(m, size):
    """Primitive (where one exists), then non-primitive: 1, an element of smaller order, and an arbitrary value >= m."""
    out = []
    w = _primitive(m, size) if m != 12 else None
    if w is not None:
        out.append(w)
        out.append(w * w % m)
    out += [1, m + 3 if m + 3 < 65536 else 5]
    return out


def test_fft_restatement_matches_the_oracle(oracle):
    rng = np.random.default_rng(4)
    for m in (17, 257, 337):
        for size in SIZES:
            for omega in sorted(set(omegas(m, size) + [0, m - 1])):
                x = rng.integers(0, 65536, size=(size, 3), dtype=np.int64)
                for inverse in (False, True):
                    want = ref_fft(x, m, omega, inverse)
                    for i in range(3):
                        assert oracle.fft(m, omega, size, "cooley_tukey", inverse, [int(v) for v in x[:, i]]) == want[:, i].tolist(), (m, size, omega, inverse)
            for la in sorted({1, size // 2, size - 1} - {0}):
                a = rng.integers(0, 65536, size=(la, 5), dtype=np.uint16)
                b = rng.integers(0, 65536, size=(size - la, 5), dtype=np.uint16)
                for omega in omegas(m, size):
                    assert np.array_equal(ref_mul_ntt(a.astype(np.int64), b.astype(np.int64), m, omega),
                                          oracle.mul_ntt_batch(a, b, m, omega)), (m, size, la, omega)
    with pytest.raises(ArithmeticError):
        ref_fft(np.ones((4, 1), np.int64), 2, 1, inverse=True)
    assert ref_fft(np.array([[1], [1]]), 2, 1).tolist() == [[0], [0]]


def _u16(rng, shape):
    x = rng.integers(0, 65536, size=shape, dtype=np.uint16)
    x[:, :7] = 0xFFFF
    x[:, 7:11] = 0
    return x


def ntt_call(ctx, n, m, omega, size, inverse, i, o, dev):
    return ctx.lib.pbh_ntt_generic_batch(ctx.h, C.c_size_t(n), C.c_uint32(m), C.c_uint32(omega), C.c_uint32(size), int(inverse),
                                         *_pp(i), *_pp(o), int(dev))


def mul_call(ctx, n, m, omega, la, lb, a, b, o, dev):
    return ctx.lib.pbh_mul_ntt_batch(ctx.h, C.c_size_t(n), C.c_uint32(m), C.c_uint32(omega), C.c_uint32(la), C.c_uint32(lb),
                                     *_pp(a), *_pp(b), *_pp(o), int(dev))


def run_ntt(ctx, x, m, omega, inverse, dev, aligned=True, key=None):
    size, n = x.shape
    i = Buf(x, *place("in", 0, n, aligned), dev, np.uint16)
    o = Buf(None, *place("out", 0, n, aligned), dev, np.uint16, planes=size, n=n)
    try:
        want = ref_fft(x, m, omega, inverse)
    except ArithmeticError:
        want = None
    before = ctx.launch_count
    rc = []
    fn = lambda: rc.append(ntt_call(ctx, n, m, omega, size, inverse, i, o, dev)) or ctx.sync()
    if key and want is not None:
        assert_census(key, fn, ["ntt_generic_kernel"])
    else:
        fn()
    what = f"ntt m={m} size={size} omega={omega} inverse={inverse} dev={dev} n={n}"
    if want is None:
        assert rc[0] == SETUP_PANIC and ctx.launch_count == before, what
        o.check(np.full((size, n), GUARD * 0x0101, np.uint16), what)
    else:
        assert rc[0] == OK, (what, ctx.lib.pbh_last_error(ctx.h))
        o.check(want, what)
    i.untouched(what)


def run_mul(ctx, a, b, m, omega, dev, aligned=True, key=None):
    la, n = a.shape; lb = b.shape[0]
    A = Buf(a, *place("in", 0, n, aligned), dev, np.uint16); B = Buf(b, *place("in", 1, n, aligned), dev, np.uint16)
    o = Buf(None, *place("out", 0, n, aligned), dev, np.uint16, planes=la + lb, n=n)
    try:
        want = ref_mul_ntt(a.astype(np.int64), b.astype(np.int64), m, omega)
    except ArithmeticError:
        want = None
    before = ctx.launch_count
    rc = []
    fn = lambda: rc.append(mul_call(ctx, n, m, omega, la, lb, A, B, o, dev)) or ctx.sync()
    if key and want is not None:
        assert_census(key, fn, ["mul_ntt_kernel"])
    else:
        fn()
    what = f"mul_ntt m={m} la={la} lb={lb} omega={omega} dev={dev} n={n}"
    if want is None:
        assert rc[0] == SETUP_PANIC and ctx.launch_count == before, what
    else:
        assert rc[0] == OK, (what, ctx.lib.pbh_last_error(ctx.h))
        o.check(want, what)
    A.untouched(what); B.untouched(what)


@gpu
@pytest.mark.parametrize("m", MODULI)
def test_ntt_generic_and_product(gpu_ctx, profiler_ok, m):
    """Every size 2..64 with primitive and non-primitive omega, forward and inverse, inputs over the whole uint16 range,
    device pointers (aligned and odd placements) and host pointers; the product for three splits of every size."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(m)
    for size in SIZES:
        for k, omega in enumerate(omegas(m, size)):
            x = _u16(rng, (size, 263))
            for inverse in (False, True):
                run_ntt(ctx, x, m, omega, inverse, dev=k != 1, aligned=k % 2 == 0, key=("ntt", m, size, inverse) if k == 0 else None)
            for la in sorted({1, size // 2, size - 1} - {0}):
                a, b = _u16(rng, (la, 131)), _u16(rng, (size - la, 131))
                run_mul(ctx, a, b, m, omega, dev=k != 1, aligned=k % 2 == 0, key=("mul", m, size) if k == 0 else None)


@gpu
def test_ntt_modulus_two_and_even_moduli(gpu_ctx):
    """The forward transform needs no length inverse: modulus 2 and 12 compute it; their inverse and product panic."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(2)
    for m in (2, 12, 65534):
        for size in (2, 8, 64):
            x = _u16(rng, (size, 40))
            run_ntt(ctx, x, m, 1, False, dev=True)
            run_ntt(ctx, x, m, 1, True, dev=True)
            run_mul(ctx, x[:1], x[1:], m, 1, dev=True)


@gpu
def test_ntt_arguments(gpu_ctx):
    """modulus >= 2^16 or < 2, size not a power of two in [2, 64], la + lb likewise: PBH_ERR_UNSUPPORTED with no launch;
    pitch < n and null pointers: PBH_ERR_BAD_ARGUMENT."""
    ctx = gpu_ctx["table"]
    x = np.zeros((64, 10), np.uint16)
    i = Buf(x, 16, 16, True, np.uint16); o = Buf(None, 16, 16, True, np.uint16, planes=64, n=10)
    before = ctx.launch_count
    for m, size in ((65536, 4), (1 << 20, 4), (1, 4), (0, 4), (17, 3), (17, 6), (17, 1), (17, 0), (17, 128)):
        assert ntt_call(ctx, 10, m, 1, size, 0, i, o, True) == UNSUPPORTED, (m, size)
    for m, la, lb in ((65536, 2, 2), (17, 1, 2), (17, 3, 3), (17, 0, 4), (17, 4, 0), (17, 40, 24 + 64)):
        assert mul_call(ctx, 10, m, 1, la, lb, i, i, o, True) == UNSUPPORTED, (m, la, lb)
    short = Buf(None, 16, 9, True, np.uint16, planes=64, n=9)
    assert ntt_call(ctx, 10, 17, 4, 4, 0, i, short, True) == BAD_ARGUMENT
    assert ctx.lib.pbh_ntt_generic_batch(ctx.h, C.c_size_t(10), 17, 4, 4, 0, None, C.c_size_t(16), *_pp(o), 1) == BAD_ARGUMENT
    assert ctx.launch_count == before
    o.check(np.full((64, 10), GUARD * 0x0101, np.uint16), "refused calls write nothing")


@gpu
def test_ntt_past_the_grid_cap(gpu_ctx):
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(9)
    n = grid_cap() + BLOCK // 3
    run_ntt(ctx, _u16(rng, (64, n)), 12289, _primitive(12289, 64), True, dev=True, aligned=False)
    run_mul(ctx, _u16(rng, (5, n)), _u16(rng, (11, n)), 40961, _primitive(40961, 16), dev=True)


# =============================================================================================
# 3. polynomial product
# =============================================================================================
def ref_poly_mul(a, b):
    la, lb = a.shape[0], b.shape[0]
    out = np.zeros((la + lb - 1, a.shape[1]), np.int64)
    a, b = a.astype(np.int64), b.astype(np.int64)
    for i in range(la):
        for j in range(lb):
            out[i + j] += a[i] * b[j]
    return (out % 17).astype(np.uint8)


def _operands(rng, planes, n):
    """All-255 (the largest exact-FP32 sums), all-zero and uniform stretches."""
    x = rng.integers(0, 256, size=(planes, n), dtype=np.uint8)
    x[:, : n // 4] = 255
    x[:, n // 4: n // 3] = 0
    return x


def mul_kernels(la, lb, n, vec):
    """pbh_poly_mul_batch's dispatch: poly_mul_vec_kernel<LA, LB> (lengths padded to even) on n / 4 words when both
    lengths are <= 8 and every base and pitch is 4-byte aligned, poly_mul_kernel for the rest."""
    ev = lambda l: 2 * ((l + 1) // 2)
    vec = vec and la <= 8 and lb <= 8
    names = [f"poly_mul_vec_kernel<{ev(la)},{ev(lb)}>"] if vec and n >= 4 else []
    return names + (["poly_mul_kernel"] if not vec or n % 4 else [])


def run_poly_mul(ctx, a, b, dev, aligned=True, key=None):
    la, n = a.shape; lb = b.shape[0]
    A = Buf(a, *place("in", 0, n, aligned), dev); B = Buf(b, *place("in", 1, n, aligned), dev)
    o = Buf(None, *place("out", 0, n, aligned), dev, planes=la + lb - 1, n=n)
    fn = lambda: ctx._check(ctx.lib.pbh_poly_mul_batch(ctx.h, C.c_size_t(n), C.c_uint32(la), C.c_uint32(lb), *_pp(A), *_pp(B), *_pp(o),
                                                       int(dev)), "pbh_poly_mul_batch") or ctx.sync()
    if key:
        assert_census(key, fn, mul_kernels(la, lb, n, aligned and (dev or n % 4 == 0)))
    else:
        fn()
    what = f"poly_mul la={la} lb={lb} n={n} dev={dev} aligned={aligned}"
    o.check(ref_poly_mul(a, b), what)
    A.untouched(what); B.untouched(what)


@gpu
@pytest.mark.parametrize("la", range(1, 17))
def test_poly_mul_every_shape(gpu_ctx, profiler_ok, la):
    """Every lb 1..16 with this la, aligned device placements at n % 4 = 1 and 3 (vector body + general tail), an odd
    placement (general kernel only) and host staging (pitch n)."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(la)
    for lb in range(1, 17):
        for k, n in enumerate((4097, 1031)):
            run_poly_mul(ctx, _operands(rng, la, n), _operands(rng, lb, n), True, key=("mul", la, lb) if k == 0 else None)
        run_poly_mul(ctx, _operands(rng, la, 1030), _operands(rng, lb, 1030), True, aligned=False)
        run_poly_mul(ctx, _operands(rng, la, 1032), _operands(rng, lb, 1032), False, aligned=False)


@gpu
@pytest.mark.parametrize("la", (2, 4, 6, 8))
def test_poly_mul_vec_past_the_grid_cap(gpu_ctx, la):
    """For each instantiation <la, lb>: more words than the capped grid has threads, then a ragged tail of 3 items; odd
    lengths ride the same instantiation."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(100 + la)
    n = 4 * (grid_cap() + 5) + 3
    for lb in (2, 4, 6, 8):
        l1, l2 = (la, lb) if lb % 4 == 0 else (la - 1, lb - 1 or 1)
        run_poly_mul(ctx, _operands(rng, l1, n), _operands(rng, l2, n), True)


# =============================================================================================
# 4. KZG commitment across SRSs
# =============================================================================================
KZG_SRS = (4, 5, 6, 9)
KZG_SECRETS = (2, 3, 7, 44)


def kzg_kernels(algo, n, n_pts, vec):
    if algo == "arith":
        return ["kzg_commit_kernel<0>"]
    n4 = n // 4 if vec and n_pts >= 7 else 0
    return (["kzg_commit_table_vec_kernel"] if n4 else []) + (["kzg_commit_kernel<1>"] if n4 * 4 < n else [])


def _coeffs(rng, n):
    x = rng.integers(0, 256, size=(7, n), dtype=np.uint8)
    x[:, : n // 8] = 255
    x[4:, n // 8: n // 3] = rng.integers(0, 16, size=(3, n // 3 - n // 8), dtype=np.uint8) * 17   # top coefficients = 0 mod 17
    x[6, n // 3: n // 2] = 17                                                                      # degree 5 at most
    return x


def run_kzg(ctx, oracle, x, s, srs_n, dev=True, aligned=True, key=None):
    n = x.shape[1]
    i = Buf(x, *place("in", 0, n, aligned), dev)
    o = Buf(None, *place("out", 0, n, aligned), dev, planes=3, n=n)
    fn = lambda: ctx._check(ctx.lib.pbh_kzg_commit_batch(ctx.h, C.c_size_t(n), *_pp(i), *_pp(o), int(dev)), "pbh_kzg_commit_batch") or ctx.sync()
    if key:
        assert_census(key, fn, kzg_kernels(ctx.algo, n, srs_n + 1, aligned and dev))
    else:
        fn()
    what = f"kzg s={s} srs_n={srs_n} algo={ctx.algo} n={n}"
    want = oracle.kzg_commit_batch(x, s, srs_n)
    o.check(want, what)
    i.untouched(what)
    return want


@gpu
@pytest.mark.parametrize("srs_n", KZG_SRS)
def test_kzg_commit_across_srs(oracle, profiler_ok, srs_n):
    """Both algorithms against SRS::eval_at_s, including the 0xFF sentinel where the polynomial is longer than the SRS;
    n % 4 = 0..3 so that the TABLE vector body and its one-block tail both run."""
    import pbh_b200 as P
    rng = np.random.default_rng(srs_n)
    ran = 0
    for s in KZG_SECRETS:
        try:
            ctx = P.Context(s=s, srs_n=srs_n, device=0)
        except P.ReferencePanic:
            continue
        with ctx:
            for algo in ("table", "arith"):
                ctx.set_algo(algo)
                for n in (1024, 1025, 1026, 1027):
                    want = run_kzg(ctx, oracle, _coeffs(rng, n), s, srs_n, aligned=n != 1026, key=("kzg", s, srs_n, algo, n))
                    if srs_n < 6:
                        assert (want[2] == 0xFF).any()
                run_kzg(ctx, oracle, _coeffs(rng, 517), s, srs_n, dev=False)
        ran += 1
    assert ran >= 2


@gpu
def test_kzg_table_past_the_grid_cap(gpu_ctx, oracle):
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(77)
    run_kzg(ctx, oracle, _coeffs(rng, 4 * (grid_cap() + 9) + 3), 2, 6)


# =============================================================================================
# 5. general division and ragged add / subtract
# =============================================================================================
def _strip(v):
    v = [int(x) for x in v]
    while len(v) > 1 and v[-1] == 0:
        v.pop()
    return v


def _pad(v, ln):
    return v + [0] * (ln - len(v))


def _batch(rng, planes, n):
    """Bytes 0..255 (>= 17 reduced as F17::from reduces them), a zero item, items whose normalised length is shorter than
    the plane count (top planes 0 or multiples of 17)."""
    x = rng.integers(0, 256, size=(planes, n), dtype=np.uint8)
    x[:, 0] = 0
    x[:, 1] = 17 * rng.integers(0, 16, size=planes)
    if planes > 1:
        x[planes // 2:, 2:5] = 0
        x[-1, 5:7] = 34
    return x


def divrem_want(oracle, num, den):
    ln, n = num.shape; ld = den.shape[0]
    q = np.zeros((ln, n), np.uint8); r = np.zeros((ld, n), np.uint8); st = np.zeros((1, n), np.uint8)
    for i in range(n):
        try:
            qo, ro = oracle.poly_op(17, "div", _strip(num[:, i] % 17), _strip(den[:, i] % 17))
            q[:, i] = _pad(qo, ln); r[:, i] = _pad(ro, ld)
        except ArithmeticError:
            st[0, i] = 1
    return q, r, st


def run_divrem(ctx, oracle, num, den, dev=True, key=None):
    ln, n = num.shape; ld = den.shape[0]
    N = Buf(num, *place("in", 0, n, False), dev); D = Buf(den, *place("in", 1, n, False), dev)
    Q = Buf(None, *place("out", 0, n, False), dev, planes=ln, n=n); R = Buf(None, *place("out", 1, n, False), dev, planes=ld, n=n)
    S = Buf(None, *place("out", 2, n, False), dev, planes=1, n=n)
    fn = lambda: ctx._check(ctx.lib.pbh_poly_divrem_batch(ctx.h, C.c_size_t(n), C.c_uint32(ln), C.c_uint32(ld), *_pp(N), *_pp(D), *_pp(Q),
                                                          *_pp(R), C.c_void_p(S.ptr), int(dev)), "pbh_poly_divrem_batch") or ctx.sync()
    if key:
        assert_census(key, fn, ["poly_divrem_kernel"])
    else:
        fn()
    what = f"divrem ln={ln} ld={ld} n={n}"
    q, r, st = divrem_want(oracle, num, den)
    Q.check(q, what); R.check(r, what); S.check(st, what)
    N.untouched(what); D.untouched(what)
    return st


def addsub_want(oracle, a, b, subtract):
    lo = max(a.shape[0], b.shape[0])
    out = np.zeros((lo, a.shape[1]), np.uint8)
    for i in range(a.shape[1]):
        out[:, i] = _pad(oracle.poly_op(17, "sub" if subtract else "add", _strip(a[:, i] % 17), _strip(b[:, i] % 17)), lo)
    return out


def run_addsub(ctx, oracle, a, b, subtract, dev=True, key=None):
    la, n = a.shape; lb = b.shape[0]
    A = Buf(a, *place("in", 0, n, False), dev); B = Buf(b, *place("in", 1, n, False), dev)
    O = Buf(None, *place("out", 0, n, False), dev, planes=max(la, lb), n=n)
    fn = lambda: ctx._check(ctx.lib.pbh_poly_addsub_ragged_batch(ctx.h, C.c_size_t(n), C.c_uint32(la), C.c_uint32(lb), int(subtract),
                                                                 *_pp(A), *_pp(B), *_pp(O), int(dev)), "pbh_poly_addsub_ragged_batch") or ctx.sync()
    if key:
        assert_census(key, fn, ["poly_addsub_ragged_kernel"])
    else:
        fn()
    what = f"addsub la={la} lb={lb} subtract={subtract} n={n}"
    O.check(addsub_want(oracle, a, b, subtract), what)
    A.untouched(what); B.untouched(what)


@gpu
@pytest.mark.parametrize("ld", range(1, 17))
def test_divrem_every_shape(gpu_ctx, oracle, profiler_ok, ld):
    """Every ln 1..32 with this ld: zero divisors (status 1), 0 / 0, short normalised lengths, bytes >= 17."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(ld)
    for ln in range(1, 33):
        num, den = _batch(rng, ln, 11), _batch(rng, ld, 11)
        den[:, 7] = 0; num[:, 8] = 0; den[:, 8] = 17            # a non-zero numerator over zero, then 0 / 0
        st = run_divrem(ctx, oracle, num, den, key=("divrem", ln, ld) if ln == 1 else None)
        assert st[0, 7] == (1 if (num[:, 7] % 17).any() else 0) and st[0, 8] == 0


@gpu
@pytest.mark.parametrize("la", range(1, 23))
def test_addsub_every_shape(gpu_ctx, oracle, profiler_ok, la):
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(50 + la)
    for lb in range(1, 23):
        a, b = _batch(rng, la, 9), _batch(rng, lb, 9)
        for subtract in (False, True):
            run_addsub(ctx, oracle, a, b, subtract, key=("addsub", la, lb, subtract) if lb == 1 else None)


@gpu
def test_divrem_and_addsub_past_the_grid_cap(gpu_ctx, oracle):
    """Tiled oracle-checked blocks past the capped grid, ending in a ragged part of a block."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(5)
    nb = 997
    count = grid_cap() + nb // 2 + 1
    tile = lambda x: np.ascontiguousarray(np.tile(x, (1, -(-count // nb)))[:, :count])
    num, den = _batch(rng, 9, nb), _batch(rng, 4, nb)
    den[:, 20:30] = 0
    q, r, st = divrem_want(oracle, num, den)
    N, D = Buf(tile(num), 3, count + 5, True), Buf(tile(den), 7, count + 9, True)
    Q = Buf(None, 1, count + 1, True, planes=9, n=count); R = Buf(None, 5, count + 3, True, planes=4, n=count)
    S = Buf(None, 2, count, True, planes=1, n=count)
    ctx._check(ctx.lib.pbh_poly_divrem_batch(ctx.h, C.c_size_t(count), 9, 4, *_pp(N), *_pp(D), *_pp(Q), *_pp(R), C.c_void_p(S.ptr), 1), "divrem")
    ctx.sync()
    Q.check(tile(q), "divrem past the cap"); R.check(tile(r), "divrem past the cap"); S.check(tile(st), "divrem past the cap")
    a, b = _batch(rng, 13, nb), _batch(rng, 6, nb)
    want = addsub_want(oracle, a, b, True)
    A, B = Buf(tile(a), 1, count + 3, True), Buf(tile(b), 2, count + 2, True)
    O = Buf(None, 3, count + 7, True, planes=13, n=count)
    ctx._check(ctx.lib.pbh_poly_addsub_ragged_batch(ctx.h, C.c_size_t(count), 13, 6, 1, *_pp(A), *_pp(B), *_pp(O), 1), "addsub")
    ctx.sync()
    O.check(tile(want), "addsub past the cap")
    for x in (N, D, A, B):
        x.untouched("past the cap")


# =============================================================================================
# 6. record transposes
# =============================================================================================
REC_OFFSET = 64        # bytes of guard before the first record (a multiple of 16)


def _records(rng, n):
    return rng.integers(0, 256, size=(n, 32), dtype=np.uint8)


def _rec_buf(x, n, dev=True, off=REC_OFFSET):
    return Buf(x, off, 32, dev, planes=n, n=32) if x is None else Buf(x, off, 32, dev)


def witness_to_planes(ctx, n, rec, bufs):
    args = []
    for k in range(3):
        args += _pp(bufs[k]) if bufs[k] is not None else _null_pp()
    return ctx.lib.pbh_witness_records_to_planes_dev(ctx.h, C.c_size_t(n), C.c_void_p(rec.ptr), *args,
                                                     C.c_void_p(bufs[3].ptr if bufs[3] is not None else None))


def proof_to_planes(ctx, n, rec, proof, status):
    return ctx.lib.pbh_proof_records_to_planes_dev(ctx.h, C.c_size_t(n), C.c_void_p(rec.ptr), *(_pp(proof) if proof is not None else _null_pp()),
                                                   C.c_void_p(status.ptr if status is not None else None))


def planes_to_proof(ctx, n, proof, status, rec):
    return ctx.lib.pbh_proof_planes_to_records_dev(ctx.h, C.c_size_t(n), *_pp(proof), C.c_void_p(status.ptr if status is not None else None),
                                                   C.c_void_p(rec.ptr))


def record_sizes():
    return (1, 255, 257, 4099, grid_cap() + BLOCK // 2 + 5)


@gpu
def test_witness_records_to_planes(gpu_ctx, profiler_ok):
    """Every subset of null planes, pitches > n with guard bytes around every plane, sizes past the grid cap."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(61)
    for n in record_sizes():
        recs = _records(rng, n)
        R = _rec_buf(recs, n)
        want = [recs[:, :12].T, recs[:, 12:21].T, recs[:, 21:26].T, recs[:, 26][None]]
        for mask in range(16) if n < 5000 else (15, 10):
            bufs = [Buf(None, *place("out", k, n, k % 2 == 0), True, planes=p, n=n) if mask >> k & 1 else None
                    for k, p in enumerate((12, 9, 5, 1))]
            fn = lambda: ctx._check(witness_to_planes(ctx, n, R, bufs), "witness records") or ctx.sync()
            assert_census(("wrec", n == 1, mask), fn, ["witness_records_to_planes_kernel"]) if n == 1 else fn()
            for k, b in enumerate(bufs):
                if b is not None:
                    b.check(np.ascontiguousarray(want[k]), f"witness records n={n} mask={mask} plane set {k}")
            R.untouched("witness records")


@gpu
def test_proof_records_round_trip(gpu_ctx, profiler_ok):
    """records -> planes (every subset of null planes) -> records: proof bytes and status come back, the reserved bytes
    are written as zero, and a null status plane writes status 0."""
    ctx = gpu_ctx["table"]
    rng = np.random.default_rng(62)
    for n in record_sizes():
        recs = _records(rng, n)
        R = _rec_buf(recs, n)
        for mask in range(4):
            proof = Buf(None, *place("out", 0, n, mask != 2), True, planes=27, n=n) if mask & 1 else None
            status = Buf(None, *place("out", 1, n, False), True, planes=1, n=n) if mask & 2 else None
            fn = lambda: ctx._check(proof_to_planes(ctx, n, R, proof, status), "proof records") or ctx.sync()
            assert_census(("prec", mask), fn, ["proof_records_to_planes_kernel"]) if n == 1 else fn()
            if proof is not None:
                proof.check(np.ascontiguousarray(recs[:, :27].T), f"proof records n={n}")
                proof.settle()
            if status is not None:
                status.check(recs[:, 27][None], f"proof records status n={n}")
                status.settle()
            R.untouched("proof records")
            if proof is None:
                continue
            for with_status in ((True, False) if status is not None else (False,)):
                out = _rec_buf(None, n, off=REC_OFFSET + 32)
                fn = lambda: ctx._check(planes_to_proof(ctx, n, proof, status if with_status else None, out), "planes to records") or ctx.sync()
                assert_census(("prec_back", with_status), fn, ["proof_planes_to_records_kernel"]) if n == 1 else fn()
                want = recs.copy()
                want[:, 28:] = 0
                if not with_status:
                    want[:, 27] = 0
                out.check(want, f"planes to records n={n} status={with_status}")
                proof.untouched("planes to records")
                if status is not None:
                    status.untouched("planes to records")


@gpu
def test_record_transposes_refuse_misaligned_records(gpu_ctx):
    """A record pointer 8 bytes past a 16-byte boundary is refused on the host (pbh_capi.cu checks the alignment before
    the launch): PBH_ERR_BAD_ARGUMENT, no launch, nothing written."""
    ctx = gpu_ctx["table"]
    n = 100
    for off in (REC_OFFSET + 8, REC_OFFSET + 4):
        R = _rec_buf(_records(np.random.default_rng(off), n), n, off=off)
        wit = Buf(None, 16, 112, True, planes=12, n=n)
        proof = Buf(None, 16, 112, True, planes=27, n=n)
        proof_in = Buf(np.zeros((27, n), np.uint8), 16, 112, True)
        before = ctx.launch_count
        assert witness_to_planes(ctx, n, R, [wit, None, None, None]) == BAD_ARGUMENT
        assert proof_to_planes(ctx, n, R, proof, None) == BAD_ARGUMENT
        assert planes_to_proof(ctx, n, proof_in, None, R) == BAD_ARGUMENT
        assert ctx.launch_count == before
        ctx.sync()
        wit.check(np.full((12, n), GUARD, np.uint8), "misaligned")
        proof.check(np.full((27, n), GUARD, np.uint8), "misaligned")
        R.untouched("misaligned")


# =============================================================================================
# 7. census bookkeeping
# =============================================================================================
@gpu
def test_census_saw_every_kernel_of_this_file(profiler_ok):
    """Runs after the cases above: the traced first calls covered all 16 poly_mul_vec_kernel instantiations and every
    other kernel this file owns."""
    if not profiler_ok:
        pytest.skip("the profiler recorded no kernel of a plain torch control kernel: no launch census on this machine")
    seen = {k for key, names in CENSUS.items() if key != "_profiler_works" for k in names}
    if len([k for k in CENSUS if k != "_profiler_works"]) < 100:
        pytest.skip("run with the rest of this file")
    want = {f"poly_mul_vec_kernel<{a},{b}>" for a in (2, 4, 6, 8) for b in (2, 4, 6, 8)} | {
        "poly_mul_kernel", "generate_kernel", "ntt_generic_kernel", "mul_ntt_kernel", "kzg_commit_table_vec_kernel", "kzg_commit_kernel<0>",
        "kzg_commit_kernel<1>", "poly_divrem_kernel", "poly_addsub_ragged_kernel", "witness_records_to_planes_kernel",
        "proof_records_to_planes_kernel", "proof_planes_to_records_kernel"}
    assert want <= seen, sorted(want - seen)
