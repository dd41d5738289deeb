"""The F_17 sweep kernels on every access path their dispatch can take, and the one-item-per-thread curve / GT sweeps past
one grid-stride pass.

pbh_capi.cu picks a sweep's access width from the bases and pitches it is given: 128-bit words (16 items per thread and
plane) when all of them are multiples of 16, 32-bit words (4 items) when they are multiples of 4, single bytes otherwise.
Poly add / sub and the division by Z_H have no 128-bit path.  Host-pointer calls stage their planes with pitch n, so
there n mod 16 decides.  Grids are capped at sm_count * per_sm blocks of 256 threads (grid_for) and loop grid-stride past
that, which only batches of millions of items reach.

The F_17 sweeps are checked against the plain numpy restatements below (pinned once against the oracle), with
guard-filled buffers around every input and output: nothing outside the n items of each plane may change, and the inputs
must come back untouched.  The curve and GT sweeps have no reference fast enough for 300 000+ items, so an oracle-checked
exhaustive block is tiled past the grid cap instead.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GUARD = 0xA5
BLOCK = 256                                   # kBlock of pbh_kernels.cuh: threads per block of every sweep
CLASSES = ("V16", "V4", "B", "mixed")         # mixed: inputs placed as V16, outputs as V4
SMALL_N = (1, 3, 4, 15, 16, 17) + tuple(4097 + r for r in range(16))
LENS = (1, 2, 7, 8, 9, 22)                    # around kAhead = 4 / 8 of poly_unary_vec and the 8-plane groups of poly_add_kernel
KINDS = ("uniform", "carry", "zero")
LARGE_N = (1 << 23) + 13


# ---------------------------------------------------------------------------------------------
# exact references: plain numpy integer code, every input byte reduced first as F17::from does
# ---------------------------------------------------------------------------------------------
def _f17(x):
    return np.asarray(x).astype(np.int64) % 17


def ntt4_matrix(k, inverse=False):
    """Forward: row i evaluates at the coset point k 4^i, M[i][j] = (k 4^i)^j.  Inverse: 13 k^-j 4^-ij (13 = 1/4)."""
    m = np.array([[pow(k * pow(4, i, 17), j, 17) for j in range(4)] for i in range(4)], dtype=np.int64)
    if not inverse:
        return m
    inv = np.array([[13 * pow(k, -j, 17) * pow(4, -i * j, 17) % 17 for i in range(4)] for j in range(4)], dtype=np.int64)
    assert ((inv @ m) % 17 == np.eye(4, dtype=np.int64)).all()
    return inv


def ref_ntt4(x, k=1, inverse=False):
    m = ntt4_matrix(k, inverse)
    c = [_f17(x[j]) for j in range(4)]
    return np.stack([(sum(int(m[i, j]) * c[j] for j in range(4)) % 17).astype(np.uint8) for i in range(4)])


def ref_add(a, b, subtract=False):
    sign = -1 if subtract else 1
    return np.stack([((_f17(a[k]) + sign * _f17(b[k])) % 17).astype(np.uint8) for k in range(a.shape[0])])


def ref_div_zh(p):
    """Long division of 22 coefficients by x^4 - 1: p = q (x^4 - 1) + r, so q_j = p_(j+4) + q_(j+4) and r_j = p_j + q_j."""
    q = [None] * 18
    for j in range(17, -1, -1):
        q[j] = ((_f17(p[j + 4]) + (q[j + 4] if j + 4 < 18 else 0)) % 17).astype(np.uint8)
    r = [((_f17(p[j]) + q[j]) % 17).astype(np.uint8) for j in range(4)]
    return np.stack(q), np.stack(r)


def ref_scale(arr):
    x = _f17(arr[-1])
    return np.stack([(_f17(a) * x % 17).astype(np.uint8) for a in arr[:-1]])


def ref_eval(arr):
    """Horner from the top coefficient down."""
    x = _f17(arr[-1])
    acc = np.zeros_like(x)
    for a in arr[-2::-1]:
        acc = (acc * x + _f17(a)) % 17
    return acc.astype(np.uint8)


def ref_div_linear(arr):
    """Synthetic division by x - c: quotient coefficients 0 .. len-2, then the remainder p(c) in plane len-1."""
    ln = arr.shape[0] - 1
    c = _f17(arr[-1])
    out = np.empty((ln, arr.shape[1]), np.uint8)
    acc = np.zeros_like(c)
    for k in range(ln - 1, -1, -1):
        if k + 1 < ln:
            out[k] = acc
        acc = (acc * c + _f17(arr[k])) % 17
    out[ln - 1] = acc
    return out


# ---------------------------------------------------------------------------------------------
# the sweeps: planes in and out, the C entry point, the reference, the dispatch widths
# ---------------------------------------------------------------------------------------------
class Sweep:
    def __init__(self, ins, outs, call, ref, widths, per_sm, zero, lens=(None,), out_pitched=True):
        self.ins, self.outs, self.call, self.ref = ins, outs, call, ref     # ins / outs: ln -> planes of each buffer
        self.widths = widths          # access widths of the dispatch, widest first
        self.per_sm = per_sm          # grid_for(ctx, ., per_sm) of the entry point
        self.zero = zero              # ln -> (input buffer, planes) that the "zero" kind fills with residue 0
        self.lens = lens
        self.out_pitched = out_pitched  # poly eval writes one plane and takes no output pitch


def _ntt_call(fn, k=None):
    def call(ctx, n, ln, i, o, dev):
        pre = () if k is None else (C.c_uint32(k),)
        return getattr(ctx.lib, fn)(ctx.h, C.c_size_t(n), *pre, *_pp(i[0]), *_pp(o[0]), int(dev))
    return call


def _unary_call(fn):
    def call(ctx, n, ln, i, o, dev):
        out = _pp(o[0]) if fn != "pbh_poly_eval_batch" else (C.c_void_p(o[0].ptr),)
        return getattr(ctx.lib, fn)(ctx.h, C.c_size_t(n), C.c_uint32(ln), *_pp(i[0]), *out, int(dev))
    return call


def _add_call(subtract):
    def call(ctx, n, ln, i, o, dev):
        return ctx.lib.pbh_poly_add_batch(ctx.h, C.c_size_t(n), C.c_uint32(ln), int(subtract), *_pp(i[0]), *_pp(i[1]), *_pp(o[0]), int(dev))
    return call


def _zh_call(ctx, n, ln, i, o, dev):
    return ctx.lib.pbh_poly_div_zh_batch(ctx.h, C.c_size_t(n), *_pp(i[0]), *_pp(o[0]), *_pp(o[1]), int(dev))


_NTT = dict(ins=lambda ln: [4], outs=lambda ln: [4], widths=(16, 4), per_sm=8, zero=lambda ln: (0, slice(1, 4, 2)))
_UNARY = dict(ins=lambda ln: [ln + 1], widths=(16, 4), per_sm=8, zero=lambda ln: (0, slice(ln, ln + 1)), lens=LENS)
_ADD = dict(ins=lambda ln: [ln, ln], outs=lambda ln: [ln], widths=(4,), per_sm=16, zero=lambda ln: (1, slice(None)), lens=LENS)
SWEEPS = {
    "ntt4": Sweep(call=_ntt_call("pbh_ntt4_batch"), ref=lambda x, ln: [ref_ntt4(x[0])], **_NTT),
    "intt4": Sweep(call=_ntt_call("pbh_intt4_batch"), ref=lambda x, ln: [ref_ntt4(x[0], 1, True)], **_NTT),
    "coset_ntt4_k2": Sweep(call=_ntt_call("pbh_coset_ntt4_batch", 2), ref=lambda x, ln: [ref_ntt4(x[0], 2)], **_NTT),
    "coset_ntt4_k3": Sweep(call=_ntt_call("pbh_coset_ntt4_batch", 3), ref=lambda x, ln: [ref_ntt4(x[0], 3)], **_NTT),
    "coset_intt4_k2": Sweep(call=_ntt_call("pbh_coset_intt4_batch", 2), ref=lambda x, ln: [ref_ntt4(x[0], 2, True)], **_NTT),
    "coset_intt4_k3": Sweep(call=_ntt_call("pbh_coset_intt4_batch", 3), ref=lambda x, ln: [ref_ntt4(x[0], 3, True)], **_NTT),
    "poly_add": Sweep(call=_add_call(False), ref=lambda x, ln: [ref_add(x[0], x[1])], **_ADD),
    "poly_sub": Sweep(call=_add_call(True), ref=lambda x, ln: [ref_add(x[0], x[1], True)], **_ADD),
    "poly_div_zh": Sweep(ins=lambda ln: [22], outs=lambda ln: [18, 4], call=_zh_call, ref=lambda x, ln: list(ref_div_zh(x[0])), widths=(4,),
                         per_sm=16, zero=lambda ln: (0, slice(18, 22))),
    "poly_scale": Sweep(outs=lambda ln: [ln], call=_unary_call("pbh_poly_scale_batch"), ref=lambda x, ln: [ref_scale(x[0])], **_UNARY),
    "poly_eval": Sweep(outs=lambda ln: [1], call=_unary_call("pbh_poly_eval_batch"), ref=lambda x, ln: [ref_eval(x[0])[None]],
                       out_pitched=False, **_UNARY),
    "poly_div_linear": Sweep(outs=lambda ln: [ln], call=_unary_call("pbh_poly_div_linear_batch"), ref=lambda x, ln: [ref_div_linear(x[0])], **_UNARY),
}


def vec_class(sweep, bases, pitches):
    """The access width the entry point dispatches to (pbh_capi.cu): the widest of its widths dividing every base and
    pitch it checks, 0 for the byte loop."""
    for w in sweep.widths:
        if all(v % w == 0 for v in (*bases, *pitches)):
            return w
    return 0


def placement_class(in_vals, out_vals):
    """The named class of a placement from its bases and pitches (inputs, outputs)."""
    div = lambda vals, w: all(v % w == 0 for v in vals)
    if div(in_vals + out_vals, 16):
        return "V16"
    if div(in_vals + out_vals, 4):
        return "mixed" if div(in_vals, 16) else "V4"
    return "B"


def expected_width(sweep, cls):
    return {"V16": sweep.widths[0], "V4": 4, "mixed": 4, "B": 0}[cls]


# ---------------------------------------------------------------------------------------------
# placement: planes at a chosen offset and pitch inside a guard-filled buffer
# ---------------------------------------------------------------------------------------------
class Placed:
    """`planes` planes of `n` bytes, `pitch` bytes apart, from byte `off` of a buffer filled with GUARD (CUDA tensor or
    numpy array)."""

    def __init__(self, planes, n, off, pitch, device):
        self.planes, self.n, self.off, self.pitch, self.device = planes, n, off, pitch, device
        size = off + planes * pitch + 64
        if device:
            import torch
            self.buf = torch.full((size,), GUARD, dtype=torch.uint8, device="cuda")
            self.ptr = self.buf.data_ptr() + off
            assert self.buf.data_ptr() % 256 == 0
        else:
            self.buf = np.full(size, GUARD, np.uint8)
            self.ptr = self.buf.ctypes.data + off

    def view(self, buf=None):
        b = self.buf if buf is None else buf
        if self.device:
            return b.as_strided((self.planes, self.n), (self.pitch, 1), self.off)
        return np.lib.stride_tricks.as_strided(b[self.off:], shape=(self.planes, self.n), strides=(self.pitch, 1))

    def write(self, x):
        if self.device:
            import torch
            self.view().copy_(torch.from_numpy(x).to(self.buf.device))
        else:
            self.view()[...] = x
        self.snapshot = self.buf.clone() if self.device else self.buf.copy()

    def read(self):
        return self.view().cpu().numpy() if self.device else self.view().copy()

    def guards_intact(self):
        """Every byte outside the planes' n items still holds GUARD: before the base, between n and the pitch, after the last plane."""
        g = self.buf.clone() if self.device else self.buf.copy()
        if self.device:
            self.view(g).fill_(GUARD)
        else:
            self.view(g)[...] = GUARD
        return bool((g == GUARD).all())

    def unchanged(self):
        if self.device:
            import torch
            return torch.equal(self.buf, self.snapshot)
        return np.array_equal(self.buf, self.snapshot)


def _pp(p):
    return C.c_void_p(p.ptr), C.c_size_t(p.pitch)


def layout(cls, role, slot, n):
    """(offset, pitch) of input or output buffer `slot` in a placement class.  Every buffer gets its own pitch, so no
    output pitch equals an input pitch."""
    room = -(-n // 16) * 16 + 32 * (slot + 1) + (16 if role == "out" else 0)
    if cls == "V16" or (cls == "mixed" and role == "in"):
        return 16 * (slot + 1), room
    if cls in ("V4", "mixed"):
        return (4, room + 8) if role == "in" else (8, room + 4)
    return (1, room) if role == "in" else (16, room + 3)              # B: unaligned input bases, unaligned output pitches


def _bytes(rng, shape, kind):
    planes, n = shape
    if kind == "uniform":
        return rng.integers(0, 256, size=shape, dtype=np.uint8)
    if kind == "carry":       # each 32-bit word of four items holds 255 in all lanes or 16 in all lanes
        w = rng.choice(np.array([255, 16], np.uint8), size=(planes, -(-n // 4)))
        return np.ascontiguousarray(np.repeat(w, 4, axis=1)[:, :n])
    assert kind == "zero"     # residue 0 in every byte: 0, 17, ..., 255
    return (rng.integers(0, 16, size=shape, dtype=np.uint8) * 17).astype(np.uint8)


def make_inputs(sweep, n, ln, kind, rng):
    """Input planes of one call.  "zero" puts residue 0 in the operand planes only (scale by 0, evaluate at 0, divide by x;
    b = 0; odd NTT coefficients; the top of the ÷Z_H numerator); "mixed" is uniform, carry and zero in three stretches."""
    xs = [_bytes(rng, (planes, n), "uniform" if kind in ("zero", "mixed") else kind) for planes in sweep.ins(ln)]
    buf, planes = sweep.zero(ln)
    if kind == "zero":
        xs[buf][planes] = _bytes(rng, xs[buf][planes].shape, "zero")
    elif kind == "mixed":
        b1, b2 = n // 3 // 16 * 16, 2 * n // 3 // 16 * 16
        for x in xs:
            x[:, b1:b2] = _bytes(rng, (x.shape[0], b2 - b1), "carry")
        xs[buf][planes, b2:] = _bytes(rng, xs[buf][planes, b2:].shape, "zero")
    return xs


def run_sweep(ctx, name, n, ln, cls, xs, exp, device=True):
    """One call on placed buffers: output == reference, every guard byte intact, inputs unchanged.  Returns the width the
    dispatch took, from the real bases and pitches of the call."""
    import torch
    sweep = SWEEPS[name]
    ins = [Placed(x.shape[0], n, *layout(cls, "in", s, n), device) for s, x in enumerate(xs)]
    for p, x in zip(ins, xs):
        p.write(x)
    outs = [Placed(planes, n, *layout(cls, "out", s, n), device) for s, planes in enumerate(sweep.outs(ln))]
    out_pitches = [p.pitch for p in outs] if sweep.out_pitched else []
    if device:
        torch.cuda.synchronize()
        width = vec_class(sweep, [p.ptr for p in ins + outs], [p.pitch for p in ins] + out_pitches)
        assert placement_class([p.ptr for p in ins] + [p.pitch for p in ins], [p.ptr for p in outs] + out_pitches) == cls
    else:
        width = vec_class(sweep, [0], [n])      # staged planes: fresh device allocations with pitch n
    rc = sweep.call(ctx, n, ln, ins, outs, device)
    assert rc == 0, ctx.lib.pbh_last_error(ctx.h)
    ctx.sync()
    for s, (o, e) in enumerate(zip(outs, exp)):
        got = o.read()
        if not np.array_equal(got, e):
            bad = np.argwhere(got != e)
            raise AssertionError(f"{name} n={n} len={ln} {cls} width={width}: output {s} differs at {len(bad)} bytes, "
                                 f"first (plane, item) {tuple(bad[0])}: got {got[tuple(bad[0])]}, want {e[tuple(bad[0])]}")
    for what, bufs in (("input", ins), ("output", outs)):
        for s, p in enumerate(bufs):
            assert p.guards_intact(), f"{name} n={n} len={ln} {cls}: guard bytes of {what} {s} overwritten"
    for s, p in enumerate(ins):
        assert p.unchanged(), f"{name} n={n} len={ln} {cls}: input {s} modified"
    return width


# ---------------------------------------------------------------------------------------------
# the references, pinned once against the oracle
# ---------------------------------------------------------------------------------------------
def test_references_match_oracle(oracle):
    rng = np.random.default_rng(1)
    n = 2000
    x = rng.integers(0, 256, size=(4, n), dtype=np.uint8)
    x[:, :300] = _bytes(rng, (4, 300), "carry"); x[:, 300:400] = 0
    assert np.array_equal(ref_ntt4(x), oracle.ntt4_batch(x))
    assert np.array_equal(ref_ntt4(x, inverse=True), oracle.intt4_batch(x))
    for k in (1, 2, 3):
        ev, co = ref_ntt4(x, k), ref_ntt4(x, k, inverse=True)
        for i in range(4):
            point = np.full((1, n), k * pow(4, i, 17) % 17, np.uint8)
            assert np.array_equal(ev[i], oracle.poly_eval_batch(np.concatenate([x, point]))), (k, i)
            assert np.array_equal(oracle.poly_eval_batch(np.concatenate([co, point])), x[i] % 17), (k, i)
    for ln in LENS:
        a, b = (rng.integers(0, 256, size=(ln, n), dtype=np.uint8) for _ in range(2))
        b[:, :200] = 0
        for sub in (False, True):
            assert np.array_equal(ref_add(a, b, sub), oracle.poly_add_batch(a, b, subtract=sub)), (ln, sub)
        arr = rng.integers(0, 256, size=(ln + 1, n), dtype=np.uint8)
        arr[ln, :300] = _bytes(rng, (1, 300), "zero")
        assert np.array_equal(ref_scale(arr), oracle.poly_scale_batch(arr)), ln
        assert np.array_equal(ref_eval(arr), oracle.poly_eval_batch(arr)), ln
        assert np.array_equal(ref_div_linear(arr), oracle.poly_div_linear_batch(arr)), ln
    p = rng.integers(0, 256, size=(22, n), dtype=np.uint8)
    p[18:, :500] = 0
    q, r = ref_div_zh(p)
    qo, ro = oracle.poly_div_zh_batch(p)
    assert np.array_equal(q, qo) and np.array_equal(r, ro)


# ---------------------------------------------------------------------------------------------
# every F_17 sweep on every class, ragged sizes, device pointers
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("name", list(SWEEPS))
def test_sweep_classes(gpu_ctx, name, cls):
    """Sizes 1 .. 17 and 4097 .. 4112 run every tail after the vector loops; lengths 1 .. 22 run the plane groups."""
    ctx = gpu_ctx["table"]
    sweep = SWEEPS[name]
    rng = np.random.default_rng(sorted(SWEEPS).index(name) * 16 + CLASSES.index(cls))
    for n in SMALL_N:
        for ln in sweep.lens:
            for kind in KINDS:
                xs = make_inputs(sweep, n, ln, kind, rng)
                assert run_sweep(ctx, name, n, ln, cls, xs, sweep.ref(xs, ln)) == expected_width(sweep, cls)


@pytest.mark.parametrize("name", list(SWEEPS))
def test_sweep_host_staging(gpu_ctx, name):
    """Host pointers: the planes are staged with pitch n, so n = 4112 / 4100 / 4104 / 4097 reach V16 / V4 / V4 / B; the
    host buffers themselves sit at odd offsets and pitches."""
    ctx = gpu_ctx["table"]
    sweep = SWEEPS[name]
    rng = np.random.default_rng(100 + sorted(SWEEPS).index(name))
    for n, cls in ((4112, "V16"), (4100, "V4"), (4104, "V4"), (4097, "B")):
        for ln in sweep.lens:
            for kind in KINDS:
                xs = make_inputs(sweep, n, ln, kind, rng)
                assert run_sweep(ctx, name, n, ln, "B", xs, sweep.ref(xs, ln), device=False) == expected_width(sweep, cls)


@pytest.mark.parametrize("name", list(SWEEPS))
def test_sweep_grid_stride(gpu_ctx, name):
    """n = 2^23 + 13 on every class: more vector words (or bytes) than the grid has threads, so blocks loop grid-stride,
    followed by a ragged tail."""
    import torch
    ctx = gpu_ctx["table"]
    sweep = SWEEPS[name]
    ln = max(sweep.lens) if sweep.lens[0] is not None else None
    cap = torch.cuda.get_device_properties(0).multi_processor_count * sweep.per_sm * BLOCK
    rng = np.random.default_rng(200 + sorted(SWEEPS).index(name))
    xs = make_inputs(sweep, LARGE_N, ln, "mixed", rng)
    exp = sweep.ref(xs, ln)
    for cls in CLASSES:
        w = expected_width(sweep, cls)
        assert -(-LARGE_N // max(w, 1)) > cap, (cls, cap)
        assert run_sweep(ctx, name, LARGE_N, ln, cls, xs, exp) == w
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# curve and GT sweeps (one item per thread) past one grid pass: oracle-checked blocks, tiled
# ---------------------------------------------------------------------------------------------
def _tiled(block, count):
    return np.ascontiguousarray(np.tile(block, (1, -(-count // block.shape[1])))[:, :count])


def test_curve_and_gt_sweeps_grid_stride(gpu_ctx, oracle):
    import torch
    ctx = gpu_ctx["arith"]
    cap = torch.cuda.get_device_properties(0).multi_processor_count * 8 * BLOCK
    pts = [(x, y, 0) for x in range(101) for y in range(101) if (y * y - x * x * x - 3) % 101 == 0] + [(0, 0, 1)]
    P = np.array(pts, dtype=np.uint8)
    add = np.ascontiguousarray(np.concatenate([np.repeat(P, 102, axis=0), np.tile(P, (102, 1))], axis=1).T)
    smul = np.ascontiguousarray(np.concatenate([np.repeat(P, 101, axis=0), np.tile(np.arange(101, dtype=np.uint8), 102)[:, None]], axis=1).T)
    g2 = [oracle.g2_mul((36, 31), k) for k in range(1, 17)]
    pair = np.ascontiguousarray(np.array([(p[0], p[1], p[2], q[0], q[1]) for p in pts + [(1, 2, 1), (48, 0, 1)] for q in g2], dtype=np.uint8).T)
    allgt = np.ascontiguousarray(np.array([(a, b) for a in range(101) for b in range(101)], dtype=np.uint8).T)
    rng = np.random.default_rng(3)
    gtm = rng.integers(0, 101, size=(4, 4000), dtype=np.uint8)
    kzg = rng.integers(0, 256, size=(7, 4000), dtype=np.uint8)
    pow600 = np.array([oracle.gt_pow((int(a), int(b)), 600) for a, b in allgt.T], dtype=np.uint8).T
    mul = np.array([oracle.gt_mul((int(a), int(b)), (int(c), int(d))) for a, b, c, d in gtm.T], dtype=np.uint8).T
    cases = (("g1_add", ctx.g1_add_batch, add, oracle.g1_add_batch(add)),
             ("g1_smul", ctx.g1_smul_batch, smul, oracle.g1_smul_batch(smul)),
             ("pairing", ctx.pairing_batch, pair, oracle.pairing_batch(pair)),
             ("gt_pow600", ctx.gt_pow600_batch, allgt, pow600),
             ("gt_mul", ctx.gt_mul_batch, gtm, mul),
             ("kzg_commit", ctx.kzg_commit_batch, kzg, oracle.kzg_commit_batch(kzg)))
    for name, fn, block, exp in cases:
        nb = block.shape[1]
        count = (cap // nb + 1) * nb + nb // 3 + 1          # whole blocks past the cap, then a ragged part of one
        assert count > cap
        got = fn(torch.from_numpy(_tiled(block, count)).cuda())
        ctx.sync()
        got = got.cpu().numpy()
        for t in range(0, count, nb):
            assert np.array_equal(got[:, t:t + nb], exp[:, :min(nb, count - t)]), (name, t // nb)


# ---------------------------------------------------------------------------------------------
# PBH_OPT_PROVER_LAUNCH_SHAPE: every instantiation of the plain-load FP32 prover gives the same bytes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", range(5))
def test_prover_launch_shapes(gpu_ctx, oracle, shape):
    """Shapes 0..4 (256 x 2, 256 x 1, 128 x 4, 128 x 5, 128 x 6 threads x resident blocks) with TMA tiles off: a seeded
    uniform batch against the oracle, and 2^20 full-path items (past every variant's grid cap) byte-equal to the default
    context."""
    import torch
    import pbh_b200
    ref = gpu_ctx["table"]
    n = 30000 + 37
    with pbh_b200.Context(device=0, algo="table") as ctx:
        ctx.set_option(pbh_b200.OPT_TMA, 0)
        ctx.set_option(pbh_b200.OPT_PROVER_LAUNCH_SHAPE, shape)
        wo, ro, co, _, _ = oracle.generate_inputs(n, seed=0x5A0 + shape, dist=0, threads=8)
        po, so = oracle.prove_batch(wo, ro, co, threads=8)
        p, s = ctx.prove_batch(*(torch.from_numpy(a).cuda() for a in (wo, ro, co)))
        ctx.sync()
        assert np.array_equal(s.cpu().numpy(), so) and np.array_equal(p.cpu().numpy(), po)
        assert set(np.unique(so)) >= {0, 2, 4, 5}
        w, r, c, _ = ref.generate_inputs(1 << 20, seed=0xB200 + shape, dist=1)
        pr, sr = ref.prove_batch(w, r, c)
        p, s = ctx.prove_batch(w, r, c)
        ctx.sync(); ref.sync()
        assert int((sr != 0).sum()) == 0
        assert torch.equal(p, pr) and torch.equal(s, sr)
