"""Every prover and verifier kernel instantiation against the oracle, at tile, warp and grid edges, with a launch census.

`INSTANTIATIONS` names each proof-system kernel the library defines together with the context settings and buffer placement
that reach it, and `expected_kernels(case)` restates the dispatch of `launch_prove`, `launch_verify`, `launch_prove_fs`,
`launch_verify_fs` and the packed Fiat-Shamir launches in pbh_capi.cu, follow-up kernels included.  The CPU test
partitions the kernels `nm` finds in the library between that table, the sweep and codec kernels other test files own and the
measurement kernels, so a kernel added without a test entry fails `-m "not gpu"`.

On the GPU each entry runs one hard corpus, built once with the oracle, at sizes derived from the SM count: ragged tiles and
warps, G - 1, G, G + 1 and 2G + 1 tiles of the persistent tile kernels' own grid G, and cap - 1 ... 2 cap + 1 blocks of the
grid-stride kernels.  Every plane sits inside guard bytes; outputs, summaries (digest, verdict bitmap, peer windows) and every
untouched byte are compared byte for byte.  The first case of each entry also runs under torch.profiler (CUDA activities
only), which asserts that exactly the expected kernels were launched."""
import os
import re
import subprocess

import numpy as np
import pytest

GUARD = 0xA5
TILE = 256
FIRST = 2**40 + 3                   # first_index of the digest: the item index does not fit 32 bits
GARBAGE = 0x5AC3_96E1_0F2D_B487     # the digest word before a call: the fused kernels overwrite it, the others zero it first
SHAPES = {0: (256, 2), 1: (256, 1), 2: (128, 4), 3: (128, 5), 4: (128, 6)}   # PBH_OPT_PROVER_LAUNCH_SHAPE -> <THREADS, MIN_BLOCKS>
SHAPE_CAP = {0: 8, 1: 8, 2: 16, 3: 20, 4: 24}                                 # blocks per SM of that launch's grid cap


def _row(kernel, op, algo, **kw):
    case = dict(kernel=kernel, op=op, algo=algo, fp32=1, vf32=0, spec=1, tma=1, shape=0, srs="pbh", aligned=True, digest=False,
                bitmap=None, peers=False, lane=False)
    for k in kw:
        assert k in case, k
    case.update(kw)
    return case


# The proof-system kernels and one way to reach each.  srs "other" is the reference circuit over SRS(7, 9): the constants no
# longer match the compiled-in ones, so the generic instantiations run.  bitmap: byte offset of the verdict bitmap mod 4.
INSTANTIATIONS = [
    # TMA provers: persistent tile kernels (prove_f32_tma_kernel<ALGO, PBH_CIRCUIT>)
    _row("prove_f32_tma_kernel<1,1>", "prove", "table"),
    _row("prove_f32_tma_kernel<1,0>", "prove", "table", srs="other"),
    _row("prove_f32_tma_kernel<0,1>", "prove", "arith"),
    _row("prove_f32_tma_kernel<0,0>", "prove", "arith", spec=0),
    _row("prove_f32_tma_kernel<1,1>", "prove", "table", digest=True, peers=True),
    _row("prove_f32_tma_kernel<0,1>", "prove", "arith", digest=True, peers=True),
    _row("prove_f32_tma_kernel<0,0>", "prove", "arith", srs="other", digest=True),
    _row("prove_f32_tma_kernel<1,1>", "prove", "table", lane=True),
    _row("prove_f32_tma_kernel<0,1>", "prove", "arith", lane=True),
    # plain-load provers: grid-stride kernels
    _row("prove_f32_kernel<0,256,2>", "prove", "arith", aligned=False),
    *[_row("prove_f32_kernel<1,%d,%d>" % SHAPES[s], "prove", "table", tma=0, shape=s) for s in SHAPES],
    _row("prove_kernel<0>", "prove", "arith", fp32=0),
    _row("prove_kernel<1>", "prove", "table", fp32=0),
    _row("digest_kernel", "prove", "table", fp32=0, digest=True),
    _row("window_publish_kernel", "prove", "arith", fp32=0, digest=True, peers=True),
    # TMA verifiers: persistent tile kernels (verify_tma_kernel<ALGO, MIN_BLOCKS, PEERS>)
    _row("verify_tma_kernel<1,4,0>", "verify", "table"),
    _row("verify_tma_kernel<1,4,0>", "verify", "table", vf32=1),
    _row("verify_tma_kernel<0,3,0>", "verify", "arith"),
    _row("verify_tma_kernel<1,4,0>", "verify", "table", bitmap=0),
    _row("verify_tma_kernel<1,4,1>", "verify", "table", bitmap=0, peers=True),
    _row("verify_tma_kernel<0,3,1>", "verify", "arith", bitmap=0, peers=True),
    _row("verify_tma_kernel<1,4,0>", "verify", "table", lane=True),
    _row("verify_tma_kernel<0,3,0>", "verify", "arith", lane=True),
    # plain-load verifiers and the bitmap fallback
    _row("verify_kernel<1>", "verify", "table", aligned=False),
    _row("verify_kernel<1>", "verify", "table", tma=0, vf32=1),
    _row("verify_kernel<0>", "verify", "arith", aligned=False),
    _row("pack_verdicts_kernel", "verify", "table", bitmap=1),
    _row("pack_verdicts_kernel", "verify", "arith", bitmap=3, peers=True),
    # Fiat-Shamir provers (prove_fs_kernel<ALGO, FP32, PBH_CIRCUIT, DIGEST>)
    _row("prove_fs_kernel<0,0,0,0>", "prove_fs", "arith", fp32=0),
    _row("prove_fs_kernel<0,1,0,0>", "prove_fs", "arith"),
    _row("prove_fs_kernel<0,1,0,1>", "prove_fs", "arith", digest=True, peers=True),
    _row("prove_fs_kernel<1,0,0,0>", "prove_fs", "table", fp32=0),
    _row("prove_fs_kernel<1,1,0,0>", "prove_fs", "table", srs="other"),
    _row("prove_fs_kernel<1,1,0,1>", "prove_fs", "table", spec=0, digest=True),
    _row("prove_fs_kernel<1,1,1,0>", "prove_fs", "table"),
    _row("prove_fs_kernel<1,1,1,1>", "prove_fs", "table", digest=True, peers=True),
    _row("digest_kernel", "prove_fs", "arith", fp32=0, digest=True),
    # Fiat-Shamir verifiers (verify_fs_kernel<ALGO, BITMAP>)
    _row("verify_fs_kernel<0,0>", "verify_fs", "arith"),
    _row("verify_fs_kernel<0,1>", "verify_fs", "arith", bitmap=0, peers=True),
    _row("verify_fs_kernel<1,0>", "verify_fs", "table"),
    _row("verify_fs_kernel<1,0>", "verify_fs", "table", vf32=1),
    _row("verify_fs_kernel<1,1>", "verify_fs", "table", bitmap=0),
    _row("pack_verdicts_kernel", "verify_fs", "table", bitmap=2, peers=True),
    # Fiat-Shamir over packed records
    _row("prove_fs_packed_kernel<0,0,0>", "prove_fs_packed", "arith", fp32=0),
    _row("prove_fs_packed_kernel<0,1,0>", "prove_fs_packed", "arith"),
    _row("prove_fs_packed_kernel<1,0,0>", "prove_fs_packed", "table", fp32=0),
    _row("prove_fs_packed_kernel<1,1,0>", "prove_fs_packed", "table", srs="other"),
    _row("prove_fs_packed_kernel<1,1,1>", "prove_fs_packed", "table"),
    _row("verify_fs_packed_kernel<0>", "verify_fs_packed", "arith"),
    _row("verify_fs_packed_kernel<1>", "verify_fs_packed", "table", vf32=1),
]

# Kernels whose paths other test files compare with the oracle: the F_17 / curve / GT sweeps (test_sweep_paths.py,
# test_gpu_parity.py, test_gpu_round2.py), the packed codecs (test_packed_format.py), and - at their path and context
# edges, with a launch census - the input generator, the generic NTT and NTT product, the polynomial product, the KZG
# commitment, the general division, the ragged add / subtract and the record transposes (test_sweep_kernel_edges.py).
SWEEP_KERNELS = sorted(
    [f"ntt4_kernel<{i},{k}>" for i in (0, 1) for k in (1, 2, 3)]
    + [f"poly_mul_vec_kernel<{a},{b}>" for a in (2, 4, 6, 8) for b in (2, 4, 6, 8)]
    + [f"poly_unary_kernel<{op}>" for op in (0, 1, 2)] + ["kzg_commit_kernel<0>", "kzg_commit_kernel<1>", "gt_kernel<0>", "gt_kernel<1>"]
    + "ntt_generic_kernel mul_ntt_kernel poly_mul_kernel poly_add_kernel poly_div_zh_kernel poly_divrem_kernel poly_addsub_ragged_kernel "
      "g1_smul_kernel g1_add_kernel kzg_commit_table_vec_kernel pairing_kernel generate_kernel witness_records_to_planes_kernel "
      "proof_records_to_planes_kernel proof_planes_to_records_kernel unpack_witness_kernel pack_proof_kernel unpack_proof_kernel".split())

# Instruction-rate probes behind pbh_measure_int32_peak: no result to compare
MEASUREMENT_KERNELS = sorted([f"int32_peak_kernel<{i}>" for i in range(8)] + [f"shift_peak_kernel<{i}>" for i in range(5)]
                             + [f"mac3_peak_kernel<{i}>" for i in (0, 1)] + [f"ffma2_peak_kernel<{i}>" for i in (0, 1)])

_KERNEL = re.compile(r"(\w+_kernel)\s*(<[^<>]*>)?\s*\(")


def normalise(symbol):
    """`family<args>` of a demangled kernel symbol (nm or CUPTI): namespace, return type, parameter list, casts and blanks
    dropped, true / false written 1 / 0.  None when the symbol is not a kernel."""
    m = _KERNEL.search(symbol)
    if not m:
        return None
    args = m.group(2) or ""
    if args:
        args = re.sub(r"\(\s*(unsigned\s+)?\w+\s*\)", "", args)          # (int)1, (bool)1
        args = re.sub(r"\s+", "", args).replace("true", "1").replace("false", "0")
        args = re.sub(r"(?<=\d)[uUlL]+", "", args)
    return m.group(1) + args


def library_kernels(lib_path):
    out = subprocess.run(["nm", "-C", "--defined-only", lib_path], check=True, capture_output=True, text=True).stdout
    names = []
    for line in out.splitlines():
        parts = line.split(None, 2)
        if len(parts) == 3 and re.match(r"^(void\s+)?pbh::\w+_kernel[<(]", parts[2]):
            names.append(normalise(parts[2]))
    return names


def expected_kernels(c):
    """The kernels one call of case `c` launches, in order: a restatement of the dispatch in pbh_capi.cu."""
    A = 1 if c["algo"] == "table" else 0
    special = c["srs"] == "pbh" and bool(c["spec"])
    publish = ["window_publish_kernel"] if c["peers"] else []
    op, bm = c["op"], c["bitmap"]
    if op == "prove":
        if c["fp32"] and c["tma"] and c["aligned"]:
            return [f"prove_f32_tma_kernel<{A},{int(special)}>"]          # digest, when asked, fused and published in the kernel
        if c["fp32"] and A == 0:
            k = "prove_f32_kernel<0,256,2>"
        elif c["fp32"]:
            k = "prove_f32_kernel<1,%d,%d>" % SHAPES.get(c["shape"], SHAPES[0])
        else:
            k = f"prove_kernel<{A}>"
        return [k] + (["digest_kernel"] + publish if c["digest"] else [])
    if op == "verify":
        tail = ["pack_verdicts_kernel"] + publish
        if c["tma"] and c["aligned"]:
            fused = bm == 0
            return [f"verify_tma_kernel<{A},{4 if A else 3},{int(fused and c['peers'])}>"] + (tail if bm not in (None, 0) else [])
        return [f"verify_kernel<{A}>"] + (tail if bm is not None else [])
    sp = int(A == 1 and bool(c["fp32"]) and special)
    if op == "prove_fs":
        fused = c["digest"] and bool(c["fp32"])
        return [f"prove_fs_kernel<{A},{int(bool(c['fp32']))},{sp},{int(fused)}>"] + (["digest_kernel"] + publish if c["digest"] and not fused else [])
    if op == "verify_fs":
        return [f"verify_fs_kernel<{A},{int(bm == 0)}>"] + (["pack_verdicts_kernel"] + publish if bm not in (None, 0) else [])
    if op == "prove_fs_packed":
        return [f"prove_fs_packed_kernel<{A},{int(bool(c['fp32']))},{sp}>"]
    if op == "verify_fs_packed":
        return [f"verify_fs_packed_kernel<{A}>"]
    raise ValueError(op)


def _row_id(c):
    flags = [k for k in ("digest", "peers", "lane") if c[k]] + ([f"bitmap{c['bitmap']}"] if c["bitmap"] is not None else [])
    flags += [f"{k}{c[k]}" for k, d in (("fp32", 1), ("vf32", 0), ("spec", 1), ("tma", 1), ("shape", 0)) if c[k] != d]
    flags += ([] if c["srs"] == "pbh" else ["srs_other"]) + ([] if c["aligned"] else ["unaligned"])
    return "-".join([c["op"], c["algo"], c["kernel"]] + flags)


# ------------------------------------------------------------------------------------------------------- the census (CPU)
def test_every_kernel_has_exactly_one_owner(product_lib):
    import pbh_b200
    found = library_kernels(pbh_b200.LIB_PATH)
    assert len(found) == len(set(found)), "a kernel symbol normalised twice"
    tested = {c["kernel"] for c in INSTANTIATIONS}
    owners = {"INSTANTIATIONS": tested, "SWEEP_KERNELS": set(SWEEP_KERNELS), "MEASUREMENT_KERNELS": set(MEASUREMENT_KERNELS)}
    for k in found:
        places = [name for name, s in owners.items() if k in s]
        assert len(places) == 1, f"{k} is listed in {places or 'no list'}: give it an entry in {__name__}.INSTANTIATIONS"
    stale = set().union(*owners.values()) - set(found)
    assert not stale, f"listed but not in the library: {sorted(stale)}"


def test_table_restates_the_dispatch():
    """Each entry's own settings reach its kernel; the kernels the entries reach are exactly the table's."""
    reached = set()
    for c in INSTANTIATIONS:
        ks = expected_kernels(c)
        assert c["kernel"] in ks, (_row_id(c), ks)
        reached |= set(ks)
        if c["lane"]:
            assert c["op"] in ("prove", "verify") and not c["digest"] and c["bitmap"] is None and not c["peers"]
    assert reached == {c["kernel"] for c in INSTANTIATIONS}
    # spot checks of the restatement against the launch code
    assert expected_kernels(_row("x", "verify", "arith", bitmap=1, peers=True)) == ["verify_tma_kernel<0,3,0>", "pack_verdicts_kernel", "window_publish_kernel"]
    assert expected_kernels(_row("x", "prove", "table", aligned=False, digest=True)) == ["prove_f32_kernel<1,256,2>", "digest_kernel"]
    assert expected_kernels(_row("x", "prove_fs", "table", spec=0, digest=True, peers=True)) == ["prove_fs_kernel<1,1,0,1>"]
    assert normalise("void pbh::verify_tma_kernel<(int)1, (int)4, true>(pbh::VerifyTmaMaps, bool)") == "verify_tma_kernel<1,4,1>"
    assert normalise("pbh::digest_kernel(unsigned long, unsigned long)") == "digest_kernel"


# ------------------------------------------------------------------------------------------------------ geometry
def tile_grid(c, sms):
    """G of the persistent tile kernels: launch_prove / launch_verify with grid_scale 2, or 1 on in-place lanes."""
    scale = 1 if c["lane"] else 2
    if c["op"] == "prove":
        return sms * scale
    if c["algo"] == "table":
        return sms * 2 * scale
    return sms * (3 if scale == 2 else 2)


def stride_grid(c):
    """(threads per block, blocks per SM of the grid cap) of a grid-stride launch."""
    k = expected_kernels(c)[0]
    if k.startswith(("prove_fs", "verify_fs")):
        return 256, 2
    if k.startswith("prove_f32_kernel<1,"):
        return SHAPES[c["shape"]][0], SHAPE_CAP[c["shape"]]
    return 256, 8


TILE_SIZES = (1, 31, 32, 33, 255, 256, 257, 272, 4096 + 16, 4096 + 17)
STRIDE_SIZES = (1, 31, 32, 33, 255, 257, 4096 + 17)


def is_tile(c):
    return c["kernel"].startswith(("prove_f32_tma_kernel", "verify_tma_kernel")) or expected_kernels(c)[0].startswith(
        ("prove_f32_tma_kernel", "verify_tma_kernel"))


def sizes_for(c, sms):
    if is_tile(c):
        G = tile_grid(c, sms)
        # a ragged last tile each time; 144 items: n % 16 == 0, the clipped tile the TMA store writes
        edges = [(G - 1, 129), (G, 144), (G + 1, 1), (2 * G + 1, 255)]
        return list(TILE_SIZES) + [(t - 1) * TILE + last for t, last in edges]
    bs, per_sm = stride_grid(c)
    cap = per_sm * sms
    return list(STRIDE_SIZES) + [(b - 1) * bs + 33 for b in (cap - 1, cap, cap + 1, 2 * cap + 1)]   # ragged last warp


def placements_for(c):
    return ("aligned", "unaligned") if is_tile(c) else ("aligned" if c["aligned"] else "unaligned",)


# ------------------------------------------------------------------------------------------------------ the corpus
# Warp types, cycled warp by warp.  Ten types over eight warps a tile put every type at every warp position of a tile; the
# ragged last warp of the sizes above falls on several of them.  Q1 compositions: which lanes of a warp of full-path items
# have a zero among the blinders b1 b3 b5 b7, so that their warp runs the Q1 scan (pbh_prove_f32.cuh) for every lane.
Q1_LANES = {
    "q1_alt": np.arange(32) % 2 == 0,
    "q1_lane0": np.arange(32) == 0,
    "q1_lane31": np.arange(32) == 31,
    "q1_all": np.ones(32, bool),
    "q1_all_but_one": np.arange(32) != 17,
    "q1_none": np.zeros(32, bool),
}
FULLPATH_POOL = 24001
WARP_TYPES = ("q1_alt", "q1_lane0", "q1_lane31", "uniform", "q1_all", "zero_blinder", "q1_all_but_one", "bad_bytes", "q1_none", "unsat")


def build_prover_inputs(oracle, n, seed, threads, s=2, srs_n=6):
    """wit (12,n), rand (9,n), chal (5,n), and the warp type of each item."""
    uw, ur, uc, _, _ = oracle.generate_inputs(n, seed=seed, dist=0, s=s, srs_n=srs_n, threads=threads)
    # full-path items are drawn by rejection, about 1000 times slower than uniform ones: a pool of them, repeated
    pool = min(n, FULLPATH_POOL)
    fw, fr, fc, _, _ = oracle.generate_inputs(pool, seed=seed + 1, dist=1, s=s, srs_n=srs_n, threads=threads)
    reps = -(-n // pool)
    fw, fr, fc = (np.tile(a, reps)[:, :n] for a in (fw, fr, fc))
    rng = np.random.default_rng(seed)
    warp = np.arange(n) // 32
    kind = np.array(WARP_TYPES)[warp % len(WARP_TYPES)]
    lane = np.arange(n) % 32
    w, r, c = fw.copy(), fr.copy(), fc.copy()
    uni = (kind == "uniform") | (kind == "zero_blinder") | (kind == "bad_bytes") | (kind == "unsat")
    w[:, uni], r[:, uni], c[:, uni] = uw[:, uni], ur[:, uni], uc[:, uni]
    us = kind == "unsat"                            # one witness value changed: a gate or a copy constraint fails
    w[lane[us] % 12, np.nonzero(us)[0]] = (w[lane[us] % 12, np.nonzero(us)[0]] + 1 + lane[us] % 16) % 17
    zb = kind == "zero_blinder"                     # the mix of test_zero_blinder_corner_cases: short polynomials, Q5 / Q15
    r[:, zb] = rng.choice(np.array([0, 0, 0, 1, 16, 5], np.uint8), size=(9, int(zb.sum())))
    c[:, zb] = rng.choice(np.array([0, 1, 16, 3, 7], np.uint8), size=(5, int(zb.sum())))
    bad = kind == "bad_bytes"                       # one byte >= 17: lanes 0-10 witness, 11-21 blinder, 22-31 challenge
    for lo, hi, plane, planes in ((0, 11, w, 12), (11, 22, r, 9), (22, 32, c, 5)):
        m = bad & (lane >= lo) & (lane < hi)
        plane[rng.integers(0, planes, int(m.sum())), np.nonzero(m)[0]] = rng.integers(17, 256, int(m.sum()))
    for name, lanes in Q1_LANES.items():
        m = (kind == name) & lanes[lane]
        r[np.array([0, 2, 4, 6])[rng.integers(0, 4, int(m.sum()))], np.nonzero(m)[0]] = 0
    return w, r, c, kind


_CURVE = None


def tamper(proof, chal, u, rng, frac=1.0):
    """The classes of test_gpu_parity._tamper, vectorised: curve points mostly outside the subgroup, off-curve coordinates,
    identity flags with and without coordinates, evaluations in and outside F_17, coordinates >= 101, stray flag bits,
    challenge bytes >= 17, z in H, several points at once.  Applied to a fraction `frac` of the items."""
    global _CURVE
    if _CURVE is None:
        _CURVE = np.array([(x, y) for x in range(101) for y in range(101) if (y * y - x * x * x - 3) % 101 == 0], np.uint8)
    p, c, uu = proof.copy(), chal.copy(), u.copy()
    n = p.shape[1]
    kind = np.where(rng.random(n) < frac, rng.integers(0, 10, n), 9)
    pt = rng.integers(0, 9, n)

    def sel(k):
        i = np.nonzero(kind == k)[0]
        return i, pt[i]

    i, q = sel(0)
    cp = _CURVE[rng.integers(0, len(_CURVE), len(i))]
    p[2 * q, i], p[2 * q + 1, i] = cp[:, 0], cp[:, 1]
    i, q = sel(1)
    p[2 * q, i], p[2 * q + 1, i] = rng.integers(0, 101, len(i)), rng.integers(0, 101, len(i))
    for k in (2, 3):
        i, q = sel(k)
        if k == 3:
            p[2 * q, i] = 0
            p[2 * q + 1, i] = 0
        lo = q < 8
        p[18, i[lo]] |= (1 << q[lo]).astype(np.uint8)
        p[19, i[~lo]] |= 1
    i, _ = sel(4)
    p[20 + rng.integers(0, 7, len(i)), i] = rng.integers(0, 17, len(i))
    i, _ = sel(5)
    p[20 + rng.integers(0, 7, len(i)), i] = rng.integers(17, 256, len(i))
    i, _ = sel(6)
    j = rng.integers(0, 4, len(i))
    a = i[j == 0]; p[rng.integers(0, 18, len(a)), a] = rng.integers(101, 256, len(a))
    a = i[j == 1]; p[19, a] |= (1 << rng.integers(1, 8, len(a))).astype(np.uint8)
    a = i[j == 2]; c[rng.integers(0, c.shape[0], len(a)), a] = rng.integers(17, 256, len(a))
    a = i[j == 3]; uu[a] = rng.integers(17, 256, len(a))
    i, _ = sel(7)
    if c.shape[0] > 3:
        c[3, i] = np.array([1, 4, 13, 16], np.uint8)[rng.integers(0, 4, len(i))]
    i, _ = sel(8)
    for _k in range(3):
        q = rng.integers(0, 9, len(i))
        cp = _CURVE[rng.integers(0, len(_CURVE), len(i))]
        p[2 * q, i], p[2 * q + 1, i] = cp[:, 0], cp[:, 1]
    return p, c, uu


def fuzz(a, rng, frac=0.02):
    a = a.copy()
    m = rng.random(a.shape) < frac
    a[m] = rng.integers(0, 256, int(m.sum()))
    return a


def by_class(n, *choices):
    """Items i with i % 3 == 0 keep choices[0], == 1 take choices[1], == 2 take choices[2] (arrays of shape (..., n))."""
    k = np.arange(n) % 3
    out = choices[0].copy()
    for j in (1, 2):
        out[..., k == j] = choices[j][..., k == j]
    return out


# ------------------------------------------------------------------------------------------------------ GPU fixtures
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def env(product_lib, oracle):
    """SM count, the corpus and its oracle outputs (on the device), and one context per configuration."""
    import torch
    import pbh_b200 as P
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    threads = os.cpu_count() or 8
    need = {}
    for c in INSTANTIATIONS:
        key = (c["op"], c["srs"])
        need[key] = max(need.get(key, 0), max(sizes_for(c, sms)))
    E = {"sms": sms, "ctx": {}, "ranks": {}, "cases": 0, "seen": {}, "census": None}
    rng = np.random.default_rng(2026)

    # byte-plane prover and verifier
    NP = max(need.get(("prove", "pbh"), 0), need.get(("verify", "pbh"), 0))
    w, r, ch, kind = build_prover_inputs(oracle, NP, 11, threads)
    u = oracle.generate_inputs(NP, seed=12, dist=0, threads=threads)[3]
    po, so = oracle.prove_batch(w, r, ch, threads=threads)
    assert {0, 1, 2, 3, 4, 32} <= set(np.unique(so).tolist()), np.unique(so)
    E["prove", "pbh"] = dict(ins=[w, r, ch], outs=[po, so])
    NO = max(need.get(("prove", "other"), 0), need.get(("prove_fs", "other"), 0), need.get(("prove_fs_packed", "other"), 0))
    w2, r2, c2, _ = build_prover_inputs(oracle, NO, 13, threads, s=7, srs_n=9)
    po2, so2 = oracle.prove_batch(w2, r2, c2, s=7, srs_n=9, threads=threads)
    assert (so2 == 0).sum() > NO // 3, np.unique(so2, return_counts=True)
    E["prove", "other"] = dict(ins=[w2, r2, c2], outs=[po2, so2])
    # verifier: honest proofs with their own challenges, tampered proofs and challenges, 2 % byte fuzz
    hp, hc = po, ch
    tp, tc, tu = tamper(hp, hc, u, rng)
    vp = by_class(NP, hp, tp, fuzz(hp, rng))
    vc = by_class(NP, hc, tc, fuzz(hc, rng))
    vu = by_class(NP, u, tu, fuzz(u, rng))
    vo, go = oracle.verify_batch(vp, vc, vu, threads=threads, want_gt=True)
    assert {0, 1, 2, 4, 0x10, 0x20} <= set(np.unique(vo).tolist()), np.unique(vo)
    E["verify", "pbh"] = dict(ins=[vp, vc, vu], outs=[vo, go])

    # Fiat-Shamir planes: the prover's witness classes (challenges are derived), tampered and fuzzed proof bytes
    for srs, (W, R, s, srs_n) in (("pbh", (w, r, 2, 6)), ("other", (w2, r2, 7, 9))):
        m = max(need.get(("prove_fs", srs), 0), need.get(("prove_fs_packed", srs), 0))
        if m == 0:
            continue
        fpo, fso, fco = oracle.prove_fs_batch(W[:, :m], R[:, :m], s=s, srs_n=srs_n, threads=threads)
        E["prove_fs", srs] = dict(ins=[W[:, :m], R[:, :m]], outs=[fpo, fso, fco])
        # packed records: the same witnesses; the bad-byte warps carry a word >= 17^7 instead
        clean_w, clean_r = np.where(W[:, :m] >= 17, 0, W[:, :m]), np.where(R[:, :m] >= 17, 0, R[:, :m])
        words = P.pack_fs_witness(clean_w, clean_r)["w"].copy()
        bad = kind[:m] == "bad_bytes" if srs == "pbh" else np.zeros(m, bool)
        words[bad, np.arange(m)[bad] % 3] = rng.integers(17**7, 2**32, int(bad.sum()), dtype=np.uint64).astype("<u4")
        ow, orr, _, _ = oracle.packed_unpack_witness(np.concatenate([words, np.zeros((m, 1), "<u4")], axis=1))
        kpo, kso, kco = oracle.prove_fs_batch(ow, orr, s=s, srs_n=srs_n, threads=threads)
        E["prove_fs_packed", srs] = dict(ins=[words], outs=[oracle.packed_pack_proofs(kpo, kso), oracle.packed_pack_chal_u(kco[:5], kco[5])])
    NF = need.get(("verify_fs", "pbh"), 0)
    fpo, fso, _ = E["prove_fs", "pbh"]["outs"]
    assert fpo.shape[1] >= NF
    dummy_c, dummy_u = np.zeros((5, NF), np.uint8), np.zeros(NF, np.uint8)
    fp = by_class(NF, fpo[:, :NF], tamper(fpo[:, :NF], dummy_c, dummy_u, rng)[0], fuzz(fpo[:, :NF], rng))
    fvo, fvc, fvg = oracle.verify_fs_batch(fp, threads=threads, want_gt=True)
    assert len(set(np.unique(fvo).tolist())) >= 4
    E["verify_fs", "pbh"] = dict(ins=[fp], outs=[fvo, fvc, fvg])
    # packed verifier: honest words, digits changed, random words and every status code (test_fs_packed_verify_of_tampered_words)
    NK = need.get(("verify_fs_packed", "pbh"), 0)
    words = oracle.packed_pack_proofs(fpo[:, :NK], fso[:NK]).copy()
    k3 = np.arange(NK) % 6
    words[k3 == 1, 0] ^= rng.integers(0, 2**32, int((k3 == 1).sum()), dtype=np.uint64).astype("<u4")
    words[k3 == 2, 1] = rng.integers(0, 2**32, int((k3 == 2).sum()), dtype=np.uint64).astype("<u4")
    words[k3 == 3, 2] = rng.integers(0, 2**29, int((k3 == 3).sum()), dtype=np.uint64).astype("<u4")
    words[k3 == 4, 2] |= ((np.arange(int((k3 == 4).sum())) % 7) + 1).astype("<u4") << 29
    words[k3 == 5] = rng.integers(0, 2**32, (int((k3 == 5).sum()), 3), dtype=np.uint64).astype("<u4")
    planes, _ = oracle.packed_unpack_proofs(words)
    kvo, _ = oracle.verify_fs_batch(planes, threads=threads)
    E["verify_fs_packed", "pbh"] = dict(ins=[words], outs=[kvo])

    for key in [k for k in E if isinstance(k, tuple)]:
        E[key]["dev_ins"] = [_dev(a if a.dtype == np.uint8 else np.ascontiguousarray(a).view(np.uint8).reshape(-1)) for a in E[key]["ins"]]
        E[key]["dev_outs"] = [_dev(a if a.dtype == np.uint8 else np.ascontiguousarray(a).view(np.uint8).reshape(-1)) for a in E[key]["outs"]]
    yield E
    torch.cuda.synchronize()
    for c in E["ctx"].values():
        c.close()
    for rk in E["ranks"].values():
        for c in rk["ctx"]:
            c.close()


def _configure(ctx, c):
    import pbh_b200 as P
    ctx.set_option(P.OPT_PROVER_FP32, c["fp32"])
    ctx.set_option(P.OPT_VERIFIER_FP32, c["vf32"])
    ctx.set_option(P.OPT_SPECIALISE, c["spec"])
    ctx.set_option(P.OPT_TMA, c["tma"])
    ctx.set_option(P.OPT_PROVER_LAUNCH_SHAPE, c["shape"])
    ctx.set_option(P.OPT_LANE_MODE, 0 if c["lane"] else 3)


def _context(E, c):
    import pbh_b200 as P
    s, srs_n = (2, 6) if c["srs"] == "pbh" else (7, 9)
    key = (c["algo"], s, srs_n, c["fp32"], c["vf32"], c["spec"], c["tma"], c["shape"], c["lane"])
    if key not in E["ctx"]:
        E["ctx"][key] = P.Context(device=0, algo=c["algo"], s=s, srs_n=srs_n)
        _configure(E["ctx"][key], c)
    return E["ctx"][key]


def _ranks(E, c):
    """Two ranks of one process on cuda:0 with a peer window each (pbh_window_attach_ptrs), one pair per configuration."""
    import pbh_b200 as P
    key = (c["algo"], c["fp32"], c["vf32"], c["spec"], c["tma"], c["shape"])
    if key not in E["ranks"]:
        biggest = max(max(sizes_for(x, E["sms"])) for x in INSTANTIATIONS)
        bpr = ((biggest + 7) // 8 + 128 + 15) // 16 * 16
        ctxs = [P.Context(device=0, algo=c["algo"]) for _ in range(2)]
        wins = []
        for rank, x in enumerate(ctxs):
            _configure(x, c)
            wins.append(x.window_create(bpr, rank, 2)[0])
        for x in ctxs:
            x.window_attach_ptrs([y._window_base for y in ctxs])
        E["ranks"][key] = {"ctx": ctxs, "win": wins}
    return E["ranks"][key]


class Planes:
    """`planes` planes of n items inside a buffer filled with GUARD: pitch >= n + 64, aligned (base and pitch multiples of 16:
    the TMA path) or not (base + 1, odd pitch: the plain path).  Device memory, or page-locked mapped host memory of `host_ctx`."""

    def __init__(self, planes, n, placement, src=None, host_ctx=None):
        import torch
        self.planes, self.n, self.host = planes, n, host_ctx
        self.off, self.pitch = (0, (n + 64 + 15) // 16 * 16) if placement == "aligned" else (1, n + 65)
        size = self.off + planes * self.pitch + 64
        if host_ctx is not None:
            self.buf = host_ctx.host_alloc(size)
            self.buf[...] = GUARD
        else:
            self.buf = torch.full((size,), GUARD, dtype=torch.uint8, device="cuda")
        self.view = self.items(self.buf)
        if src is not None:
            if host_ctx is not None:
                self.view[...] = src.cpu().numpy()
            else:
                self.view.copy_(src)
        self.before = self.buf.copy() if host_ctx is not None else self.buf.clone()

    def items(self, buf):
        """The (planes, n) items of a buffer laid out like this one ((n,) for one plane)."""
        region = buf[self.off:self.off + self.planes * self.pitch].reshape(self.planes, self.pitch)
        return region[:, :self.n] if self.planes > 1 else region[0, :self.n]

    def untouched(self):
        import torch
        return np.array_equal(self.buf, self.before) if self.host is not None else torch.equal(self.buf, self.before)

    def check(self, want, what):
        """Items [0, n) equal `want` (a device tensor); every other byte still holds GUARD."""
        import torch
        buf = torch.from_numpy(self.buf.copy()).cuda() if self.host is not None else self.buf.clone()
        got = self.items(buf)
        if not torch.equal(got, want):
            bad = (got != want).reshape(-1, self.n).any(0).nonzero()
            raise AssertionError(f"{what}: {len(bad)} items differ, the first is item {int(bad[0])}")
        self.items(buf)[...] = GUARD
        assert bool((buf == GUARD).all()), f"{what}: a byte outside the {self.n} items changed"

    def free(self):
        if self.host is not None:
            self.host.host_free(self.buf)


class Summary:
    """A digest word or a verdict bitmap inside guard bytes: a device buffer, or this rank's row of its peer window (and the
    same row of the peer's window, where the kernels store it too)."""

    def __init__(self, E, c, nbytes, fill, rank):
        import torch
        self.windows = None
        self.off = 16 + (c["bitmap"] or 0)
        if c["peers"]:
            rk = _ranks(E, c)
            self.windows = [w[rank] for w in rk["win"]]       # row `rank` of the own window and of the peer's
            for w in self.windows:
                w.fill_(GUARD)
                w[self.off:self.off + nbytes] = fill
            self.buf = self.windows[rank]
        else:
            self.buf = torch.full((self.off + nbytes + 64,), GUARD, dtype=torch.uint8, device="cuda")
            self.buf[self.off:self.off + nbytes] = fill
        self.nbytes = nbytes
        self.view = self.buf[self.off:self.off + nbytes]

    def check(self, want, what):
        import torch
        for h, buf in enumerate(self.windows or [self.buf]):
            got = buf[self.off:self.off + self.nbytes]
            assert torch.equal(got, want), f"{what} (window of rank {h})" if self.windows else what
            rest = buf.clone()
            rest[self.off:self.off + self.nbytes] = GUARD
            assert bool((rest == GUARD).all()), f"{what}: a byte around it changed"


def _garbage_bytes():
    import torch
    return torch.tensor(np.array([GARBAGE], "<u8").view(np.uint8), device="cuda")


def _digest_want(po_dev, n):
    import oracle as O
    return _dev(np.array([O.digest(po_dev[:, :n].cpu().numpy(), first_index=FIRST)], "<u8").view(np.uint8))


def run_case(E, c, n, placement, i):
    """One call of entry c on the first n corpus items; every output, summary and guard byte checked."""
    import torch
    import oracle as O
    op = c["op"]
    D = E[op, c["srs"] if op.startswith("prove") else "pbh"]
    ins, outs = D["dev_ins"], D["dev_outs"]
    rank = i % 2
    ctx = _ranks(E, c)["ctx"][rank] if c["peers"] else _context(E, c)
    host = ctx if c["lane"] else None
    tag = f"{_row_id(c)} n={n} {placement}"
    bufs, inputs = [], []

    def planes(k, n_, src=None):
        p = Planes(k, n_, placement, src, host)
        bufs.append(p)
        if src is not None:
            inputs.append(p)
        return p

    if op in ("prove", "prove_fs"):
        W, R = planes(12, n, ins[0][:, :n]), planes(9, n, ins[1][:, :n])
        Ch = planes(5, n, ins[2][:, :n]) if op == "prove" else None
        Pf, St = planes(27, n), planes(1, n)
        Cout = planes(6, n) if op == "prove_fs" else None
        dg = Summary(E, c, 8, _garbage_bytes(), rank) if c["digest"] else None
        if op == "prove":
            if c["lane"]:
                ctx.prove_batch_async(0, W.view, R.view, Ch.view, Pf.view, St.view)
                ctx.lane_sync(0)
            elif dg:
                ctx.prove_digest_batch(W.view, R.view, Ch.view, Pf.view, St.view, dg.view.view(torch.int64), first_index=FIRST)
            else:
                ctx.prove_batch(W.view, R.view, Ch.view, proof=Pf.view, status=St.view)
        elif dg:
            ctx.prove_fs_digest_batch(W.view, R.view, Pf.view, St.view, dg.view.view(torch.int64), first_index=FIRST, chal=Cout.view)
        else:
            ctx.prove_fs_batch(W.view, R.view, proof=Pf.view, status=St.view, chal=Cout.view)
        ctx.sync()
        torch.cuda.synchronize()
        Pf.check(outs[0][:, :n], tag + " proof")
        St.check(outs[1][:n], tag + " status")
        if Cout is not None:
            Cout.check(outs[2][:, :n], tag + " derived challenges")
        if dg:
            dg.check(_digest_want(outs[0], n), tag + " digest")
    elif op in ("verify", "verify_fs"):
        Pf = planes(27, n, ins[0][:, :n])
        Ch = planes(5, n, ins[1][:, :n]) if op == "verify" else None
        U = planes(1, n, ins[2][:n]) if op == "verify" else None
        Res = planes(1, n)
        want_gt = c["bitmap"] is None and i % 2 == 0
        G = planes(4, n) if want_gt else None
        Cout = planes(6, n) if op == "verify_fs" and c["bitmap"] is None else None
        bm = None
        if c["bitmap"] is not None:
            bm = Summary(E, c, (n + 7) // 8, torch.full(((n + 7) // 8,), 0xEE, dtype=torch.uint8, device="cuda"), rank)
        if op == "verify":
            if c["lane"]:
                ctx.verify_batch_async(0, Pf.view, Ch.view, U.view, Res.view, G.view if G else None)
                ctx.lane_sync(0)
            elif bm:
                ctx.verify_bitmap_batch(Pf.view, Ch.view, U.view, Res.view, bm.view)
            else:
                ctx.verify_batch(Pf.view, Ch.view, U.view, result=Res.view, gt=G.view if G else None)
        elif bm:
            ctx.verify_fs_bitmap_batch(Pf.view, Res.view, bm.view)
        else:
            ctx.verify_fs_batch(Pf.view, result=Res.view, chal=Cout.view, gt=G.view if G else None)
        ctx.sync()
        torch.cuda.synchronize()
        Res.check(outs[0][:n], tag + " result")
        gt_out = outs[1] if op == "verify" else outs[2]
        if G is not None:
            G.check(gt_out[:, :n], tag + " GT")
        if Cout is not None:
            Cout.check(outs[1][:, :n], tag + " derived challenges")
        if bm:
            bm.check(_dev(O.pack_verdicts(outs[0][:n].cpu().numpy())), tag + " bitmap")
    else:
        # packed records: 4-byte aligned device records; "unaligned" puts them 4 bytes past a 16-byte boundary
        off = 0 if placement == "aligned" else 4
        rec_in = 12
        src = ins[0][:n * rec_in]
        In = torch.full((off + n * rec_in + 64,), GUARD, dtype=torch.uint8, device="cuda")
        In[off:off + n * rec_in] = src
        before = In.clone()
        nout = 12 if op == "prove_fs_packed" else 1
        Out = torch.full((off + n * nout + 64,), GUARD, dtype=torch.uint8, device="cuda")
        Cu = torch.full((off + 4 * n + 64,), GUARD, dtype=torch.uint8, device="cuda")
        if op == "prove_fs_packed":
            ctx.prove_fs_packed(In[off:off + n * rec_in], out=Out[off:off + 12 * n], chal_u=Cu[off:off + 4 * n])
        else:
            ctx.verify_fs_packed(In[off:off + n * rec_in], result=Out[off:off + n])
        ctx.sync()
        torch.cuda.synchronize()
        assert torch.equal(In, before), tag + " input changed"
        checks = [(Out, outs[0][:n * nout], nout)] + ([(Cu, outs[1][:4 * n], 4)] if op == "prove_fs_packed" else [])
        for buf, want, width in checks:
            assert torch.equal(buf[off:off + n * width], want), tag + " records"
            rest = buf.clone()
            rest[off:off + n * width] = GUARD
            assert bool((rest == GUARD).all()), tag + " a byte around the records changed"
    for b in inputs:
        assert b.untouched(), tag + " an input byte changed"
    for b in bufs:
        b.free()
    E["cases"] += 1


# ------------------------------------------------------------------------------------------------------ the launch census
def _product_families():
    return {re.match(r"\w+", k).group(0) for k in [c["kernel"] for c in INSTANTIATIONS] + SWEEP_KERNELS + MEASUREMENT_KERNELS}


def _profiled_kernels(fn):
    """Normalised names of the kernels `fn` launched, in start order, from a CUDA-activity trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = []
    for e in prof.events():
        if getattr(e, "device_type", None) is not None and str(e.device_type).endswith("CUDA"):
            evs.append((e.time_range.start, e.name))
    return [normalise(name) or name for _, name in sorted(evs)]


def _census_available(E):
    if E["census"] is None:
        import torch
        x = torch.arange(1 << 16, device="cuda", dtype=torch.float32)
        names = _profiled_kernels(lambda: x.mul_(2.0))
        E["census"] = len(names) > 0
    return E["census"]


# ------------------------------------------------------------------------------------------------------ the matrix
@pytest.mark.gpu
@pytest.mark.parametrize("c", INSTANTIATIONS, ids=[_row_id(c) for c in INSTANTIATIONS])
def test_instantiation_matches_the_oracle(env, c):
    E = env
    fams = _product_families()
    for placement in placements_for(c):
        case = dict(c, aligned=placement == "aligned")
        for i, n in enumerate(sizes_for(c, E["sms"])):
            if i == 0 and _census_available(E):
                names = [k for k in _profiled_kernels(lambda: run_case(E, case, n, placement, i)) if re.match(r"\w+", k).group(0) in fams]
                assert names == expected_kernels(case), (_row_id(case), n, placement, names)
                for k in names:
                    E["seen"][k] = E["seen"].get(k, 0) + 1
            else:
                run_case(E, case, n, placement, i)


@pytest.mark.gpu
def test_census_covers_every_instantiation(env):
    """Runs after the matrix: every kernel of INSTANTIATIONS was seen in a trace."""
    E = env
    print(f"\n[kernel instantiations] SMs {E['sms']}, (entry, size, placement) cases {E['cases']}, profiler census "
          f"{'ran' if E['census'] else 'did not run' if E['census'] is False else 'was not reached'}")
    if E["census"] is False:
        pytest.skip("the profiler recorded no kernel of a plain torch control kernel: no launch census on this machine")
    if E["census"] is None or E["cases"] == 0:
        pytest.skip("run with the matrix of this file")
    missing = sorted({c["kernel"] for c in INSTANTIATIONS} - set(E["seen"]))
    ran = len({_row_id(c) for c in INSTANTIATIONS})
    if E["cases"] < ran:
        pytest.skip("only part of the matrix ran")
    assert not missing, f"never launched: {missing}"
