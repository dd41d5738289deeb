"""pbh_b200 — Python host side of the B200-native batched Plonk-by-hand prover / verifier.

Two layers over the C ABI of include/pbh_b200.h (libpbh_b200.so, hand-written sm_100a kernels):

* `Context` — the batch API: byte-plane numpy arrays (host pointers; H2D/D2H inside the call) or
  CUDA torch tensors (device pointers; kernels only).
* the reference's own vocabulary — `f17`, `f101`, `g1f`, `Gate`, `CopyOf`, `Constrains`, `Assigment(s)`,
  `SRS`, `Challange`, `Proof`, `Plonk.prove / Plonk.verify` — as batch-of-1 wrappers that raise
  `ReferencePanic` where the Rust crate panics (src/plonk.rs:191-650, src/constraints.rs, src/pbh/mod.rs).

There is NO CPU fallback: without the compiled extension or without a CUDA device every compute call raises.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_PKG))          # plonk-by-fingers_b200/
LIB_PATH = os.path.join(_ROOT, "libpbh_b200.so")

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)

# status / result codes of include/pbh_b200.h
ST_OK, ST_UNSATISFIED, ST_ACC_DIV0, ST_T_REMAINDER, ST_T_SLICE, ST_SRS_OOB, ST_BAD_ENCODING = 0, 1, 2, 3, 4, 5, 32
VR_ACCEPT, VR_REJECT_PAIRING, VR_NOT_ON_CURVE, VR_NOT_IN_FIELD, VR_PANIC_ZH0, VR_BAD_ENCODING = 1, 0, 2, 4, 0x10, 0x20
ALGO_ARITH, ALGO_TABLE = 0, 1
OPT_PROVER_FP32, OPT_PROVER_LAUNCH_SHAPE, OPT_TMA, OPT_CHUNK_LOG2, OPT_SPECIALISE, OPT_HOST_DIRECT, OPT_VERIFIER_FP32, OPT_LANE_MODE = 1, 2, 3, 4, 5, 6, 7, 8
OPT_HOST_STAGE, OPT_PROOF_RESIDENT = 9, 10
DIST_UNIFORM, DIST_FULLPATH = 0, 1
ERR = {0: "PBH_OK", -1: "PBH_ERR_BAD_ARGUMENT", -2: "PBH_ERR_SETUP_PANIC", -3: "PBH_ERR_CUDA", -4: "PBH_ERR_NO_DEVICE",
       -5: "PBH_ERR_UNSUPPORTED"}
PANIC_MESSAGES = {
    ST_UNSATISFIED: "assertion failed: constraints.satisfies(assigments) (src/plonk.rs:199)",
    ST_ACC_DIV0: "called `Option::unwrap()` on a `None` value (src/plonk.rs:297)",
    ST_T_REMAINDER: "assertion failed: `(left == right)` rem != Poly::zero() (src/plonk.rs:370)",
    ST_T_SLICE: "range end index 18 out of range for slice (src/plonk.rs:376)",
    ST_SRS_OOB: "index out of bounds: the len is 7 (src/plonk.rs:56)",
    ST_BAD_ENCODING: "input byte outside the field (not representable in the reference)",
}

EXPORTS = """pbh_circuit_pbh_test pbh_ctx_create pbh_ctx_destroy pbh_last_error pbh_ctx_set_algo pbh_ctx_get_algo pbh_ctx_set_option
pbh_ctx_device pbh_ctx_sync pbh_ctx_stream pbh_ctx_launch_count pbh_ctx_get_srs pbh_ctx_get_verifier_constants
pbh_prove_batch pbh_prove_batch_dev pbh_verify_batch pbh_verify_batch_dev pbh_prove_verify_batch pbh_prove_records pbh_verify_records pbh_witness_records_to_planes_dev
pbh_proof_records_to_planes_dev pbh_proof_planes_to_records_dev pbh_prove_digest_batch_dev pbh_verify_bitmap_batch_dev pbh_ntt4_batch pbh_intt4_batch
pbh_ntt_generic_batch pbh_poly_mul_batch pbh_poly_add_batch pbh_poly_div_zh_batch pbh_g1_smul_batch pbh_g1_add_batch
pbh_kzg_commit_batch pbh_pairing_batch pbh_pack_verdicts_dev pbh_digest_dev pbh_generate_inputs_dev
pbh_measure_int32_peak pbh_mul_ntt_batch pbh_poly_scale_batch pbh_poly_eval_batch pbh_poly_div_linear_batch pbh_ctx_get_fs_seed pbh_prove_fs_batch pbh_prove_fs_batch_dev pbh_verify_fs_batch pbh_verify_fs_batch_dev
pbh_prove_batch_async pbh_verify_batch_async pbh_lane_sync pbh_host_alloc pbh_host_free pbh_ctx_numa_node
pbh_coset_ntt4_batch pbh_coset_intt4_batch pbh_multi_create pbh_multi_destroy pbh_multi_device_count pbh_multi_ctx pbh_multi_last_error
pbh_multi_set_algo pbh_multi_prove_batch pbh_multi_verify_batch pbh_multi_prove_verify_sharded
pbh_gt_mul_batch pbh_gt_pow600_batch pbh_poly_divrem_batch pbh_poly_addsub_ragged_batch
pbh_prove_packed pbh_verify_packed pbh_prove_packed_async pbh_verify_packed_async pbh_prove_verify_packed pbh_unpack_witness_dev
pbh_pack_proof_dev pbh_unpack_proof_dev pbh_pack_witness_host pbh_unpack_witness_host pbh_pack_chal_u_host pbh_pack_proofs_host
pbh_unpack_proofs_host pbh_window_create pbh_window_attach pbh_window_attach_ptrs pbh_window_share pbh_window_destroy pbh_multi_prove_packed pbh_multi_verify_packed pbh_prove_verify_packed_async pbh_host_alloc_input
pbh_prove_fs_packed pbh_verify_fs_packed pbh_prove_fs_packed_async pbh_verify_fs_packed_async pbh_prove_fs_packed_dev pbh_verify_fs_packed_dev
pbh_pack_fs_witness_host pbh_unpack_fs_witness_host pbh_prove_fs_digest_batch_dev pbh_verify_fs_bitmap_batch_dev pbh_multi_prove_fs_batch
pbh_multi_verify_fs_batch pbh_multi_prove_fs_packed pbh_multi_verify_fs_packed pbh_multi_prove_verify_fs_sharded""".split()


# 32-byte records of include/pbh_b200.h
WITNESS_RECORD = np.dtype([("wit", np.uint8, (12,)), ("rand", np.uint8, (9,)), ("chal", np.uint8, (5,)), ("u", np.uint8), ("reserved", np.uint8, (5,))])
PROOF_RECORD = np.dtype([("xy", np.uint8, (18,)), ("inf_lo", np.uint8), ("inf_hi", np.uint8), ("evals", np.uint8, (7,)), ("status", np.uint8),
                         ("reserved", np.uint8, (4,))])


def witness_records(wit, rand, chal, u=None):
    """Byte planes (12,n) (9,n) (5,n) [(n,)] -> array of WITNESS_RECORD."""
    n = np.shape(wit)[1]
    rec = np.zeros(n, dtype=WITNESS_RECORD)
    rec["wit"] = np.asarray(wit).T; rec["rand"] = np.asarray(rand).T; rec["chal"] = np.asarray(chal).T
    if u is not None:
        rec["u"] = np.asarray(u)
    return rec


def proof_records(proof, status=None):
    """Byte planes (27,n) [(n,)] -> array of PROOF_RECORD."""
    proof = np.asarray(proof)
    rec = np.zeros(proof.shape[1], dtype=PROOF_RECORD)
    rec["xy"] = proof[:18].T; rec["inf_lo"] = proof[18]; rec["inf_hi"] = proof[19]; rec["evals"] = proof[20:27].T
    if status is not None:
        rec["status"] = np.asarray(status)
    return rec


def proof_planes(rec):
    """Array of PROOF_RECORD -> ((27,n) planes, (n,) status)."""
    n = rec.shape[0]
    proof = np.zeros((27, n), dtype=np.uint8)
    proof[:18] = rec["xy"].T; proof[18] = rec["inf_lo"]; proof[19] = rec["inf_hi"]; proof[20:27] = rec["evals"].T
    return proof, rec["status"].copy()


class PbhError(RuntimeError):
    """A negative return code of the C ABI."""


class ReferencePanic(RuntimeError):
    """The reference crate would panic on this input; `.status` is the PBH_ST_* / PBH_VR_* code."""

    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


class Circuit(C.Structure):
    """pbh_circuit of include/pbh_b200.h == Constrains of src/constraints.rs:109-118 for 4 gates."""
    _fields_ = [(name, C.c_uint8 * 4) for name in (
        "q_l", "q_r", "q_o", "q_m", "q_c", "c_a_wire", "c_a_index", "c_b_wire", "c_b_index", "c_c_wire", "c_c_index")]

# packed records of include/pbh_b200.h ("packed wire format"): 16-byte prover inputs, 12-byte proofs, 4-byte challenge words
PACKED_WITNESS = np.dtype([("w", "<u4", (4,))])
PACKED_PROOF = np.dtype([("points_lo", "<u4"), ("points_hi", "<u4"), ("evals_status", "<u4")])
# Fiat-Shamir prover input: wit + rand only, words 0..2 of PACKED_WITNESS
PACKED_FS_WITNESS = np.dtype([("w", "<u4", (3,))])
ST_UNREPRESENTABLE = 33


def _host_u8(a, planes, name):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim == 1:
        a = a.reshape(1, -1)
    if a.shape[0] != planes:
        raise PbhError(f"{name}: expected {planes} planes, got {a.shape[0]}")
    return a


def pack_witness(wit, rand, chal=None, u=None):
    """Byte planes (host) -> PACKED_WITNESS array (pbh_pack_witness_host: a CPU format conversion, no device involved)."""
    lib = load_library()
    W = _host_u8(wit, 12, "wit"); n = W.shape[1]
    R = _host_u8(rand, 9, "rand")
    Ch = _host_u8(chal, 5, "chal") if chal is not None else None
    U = np.ascontiguousarray(u, dtype=np.uint8).reshape(-1) if u is not None else None
    out = np.zeros(n, dtype=PACKED_WITNESS)
    rc = lib.pbh_pack_witness_host(C.c_size_t(n), C.c_void_p(W.ctypes.data), C.c_size_t(n), C.c_void_p(R.ctypes.data), C.c_size_t(n),
                                   C.c_void_p(Ch.ctypes.data if Ch is not None else None), C.c_size_t(n),
                                   C.c_void_p(U.ctypes.data if U is not None else None), C.c_void_p(out.ctypes.data))
    if rc != 0:
        raise PbhError(f"pbh_pack_witness_host: {ERR.get(rc, rc)} (a value >= 17 has no packed form)")
    return out


def unpack_witness(packed):
    """PACKED_WITNESS array -> (wit, rand, chal, u) byte planes."""
    lib = load_library()
    pk = np.ascontiguousarray(packed, dtype=PACKED_WITNESS); n = pk.shape[0]
    wit, rand, chal, u = (np.zeros((k, n), np.uint8) for k in (12, 9, 5, 1))
    rc = lib.pbh_unpack_witness_host(C.c_size_t(n), C.c_void_p(pk.ctypes.data), C.c_void_p(wit.ctypes.data), C.c_size_t(n),
                                     C.c_void_p(rand.ctypes.data), C.c_size_t(n), C.c_void_p(chal.ctypes.data), C.c_size_t(n),
                                     C.c_void_p(u.ctypes.data))
    if rc != 0:
        raise PbhError(f"pbh_unpack_witness_host: {ERR.get(rc, rc)}")
    return wit, rand, chal, u[0]


def pack_fs_witness(wit, rand):
    """Byte planes (host) -> PACKED_FS_WITNESS array (pbh_pack_fs_witness_host, a CPU format conversion)."""
    lib = load_library()
    W = _host_u8(wit, 12, "wit"); n = W.shape[1]
    R = _host_u8(rand, 9, "rand")
    if R.shape[1] != n:
        raise PbhError("wit and rand must have the same number of items")
    out = np.zeros(n, dtype=PACKED_FS_WITNESS)
    rc = lib.pbh_pack_fs_witness_host(C.c_size_t(n), C.c_void_p(W.ctypes.data), C.c_size_t(n), C.c_void_p(R.ctypes.data), C.c_size_t(n),
                                      C.c_void_p(out.ctypes.data))
    if rc != 0:
        raise PbhError(f"pbh_pack_fs_witness_host: {ERR.get(rc, rc)} (a value >= 17 has no packed form)")
    return out


def unpack_fs_witness(packed):
    """PACKED_FS_WITNESS array -> (wit, rand) byte planes."""
    lib = load_library()
    pk = np.ascontiguousarray(packed, dtype=PACKED_FS_WITNESS); n = pk.shape[0]
    wit, rand = np.zeros((12, n), np.uint8), np.zeros((9, n), np.uint8)
    rc = lib.pbh_unpack_fs_witness_host(C.c_size_t(n), C.c_void_p(pk.ctypes.data), C.c_void_p(wit.ctypes.data), C.c_size_t(n),
                                        C.c_void_p(rand.ctypes.data), C.c_size_t(n))
    if rc != 0:
        raise PbhError(f"pbh_unpack_fs_witness_host: {ERR.get(rc, rc)}")
    return wit, rand


def pack_chal_u(chal, u):
    lib = load_library()
    Ch = _host_u8(chal, 5, "chal"); n = Ch.shape[1]
    U = np.ascontiguousarray(u, dtype=np.uint8).reshape(-1)
    out = np.zeros(n, dtype="<u4")
    rc = lib.pbh_pack_chal_u_host(C.c_size_t(n), C.c_void_p(Ch.ctypes.data), C.c_size_t(n), C.c_void_p(U.ctypes.data), C.c_void_p(out.ctypes.data))
    if rc != 0:
        raise PbhError(f"pbh_pack_chal_u_host: {ERR.get(rc, rc)} (a value >= 17 has no packed form)")
    return out


def pack_proofs(proof, status=None):
    """(27, n) proof planes (+ status) -> PACKED_PROOF array; inexpressible proofs get status code 6 (ST_UNREPRESENTABLE)."""
    lib = load_library()
    P = _host_u8(proof, 27, "proof"); n = P.shape[1]
    S = np.ascontiguousarray(status, dtype=np.uint8).reshape(-1) if status is not None else None
    out = np.zeros(n, dtype=PACKED_PROOF)
    rc = lib.pbh_pack_proofs_host(C.c_size_t(n), C.c_void_p(P.ctypes.data), C.c_size_t(n), C.c_void_p(S.ctypes.data if S is not None else None),
                                  C.c_void_p(out.ctypes.data))
    if rc != 0:
        raise PbhError(f"pbh_pack_proofs_host: {ERR.get(rc, rc)}")
    return out


def unpack_proofs(packed):
    """PACKED_PROOF array -> ((27, n) proof planes, status)."""
    lib = load_library()
    pk = np.ascontiguousarray(packed, dtype=PACKED_PROOF); n = pk.shape[0]
    proof = np.zeros((27, n), np.uint8); status = np.zeros(n, np.uint8)
    rc = lib.pbh_unpack_proofs_host(C.c_size_t(n), C.c_void_p(pk.ctypes.data), C.c_void_p(proof.ctypes.data), C.c_size_t(n), C.c_void_p(status.ctypes.data))
    if rc != 0:
        raise PbhError(f"pbh_unpack_proofs_host: {ERR.get(rc, rc)}")
    return proof, status


_LIB = None


def load_library():
    """Load libpbh_b200.so; fails loudly when it has not been built (there is no fallback)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise PbhError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(or `make -C plonk-by-fingers_b200`). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        lib.pbh_last_error.restype = C.c_char_p
        lib.pbh_last_error.argtypes = [C.c_void_p]
        lib.pbh_ctx_stream.restype = C.c_void_p
        lib.pbh_ctx_stream.argtypes = [C.c_void_p]
        lib.pbh_ctx_launch_count.restype = C.c_uint64
        lib.pbh_ctx_launch_count.argtypes = [C.c_void_p]
        lib.pbh_ctx_destroy.argtypes = [C.c_void_p]
        lib.pbh_ctx_destroy.restype = None
        lib.pbh_ctx_numa_node.argtypes = [C.c_void_p]
        lib.pbh_multi_destroy.argtypes = [C.c_void_p]
        lib.pbh_multi_destroy.restype = None
        lib.pbh_multi_device_count.argtypes = [C.c_void_p]
        lib.pbh_multi_last_error.argtypes = [C.c_void_p]
        lib.pbh_multi_last_error.restype = C.c_char_p
        lib.pbh_multi_ctx.argtypes = [C.c_void_p, C.c_int]
        lib.pbh_multi_ctx.restype = C.c_void_p
        lib.pbh_multi_set_algo.argtypes = [C.c_void_p, C.c_int]
        lib.pbh_lane_sync.argtypes = [C.c_void_p, C.c_int]
        lib.pbh_host_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        if hasattr(lib, "pbh_host_alloc_input"):
            lib.pbh_host_alloc_input.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        lib.pbh_host_free.argtypes = [C.c_void_p, C.c_void_p]
        _LIB = lib
    return _LIB


def pbh_test_circuit():
    c = Circuit()
    load_library().pbh_circuit_pbh_test(C.byref(c))
    return c


def _is_torch(x):
    return type(x).__module__.startswith("torch")


class _Planes:
    """Uniform view of a (planes, n) uint8 batch living on the host (numpy) or the device (torch)."""

    def __init__(self, arr, planes, n=None, name="array", out=False):
        self.dev = _is_torch(arr)
        if self.dev:
            import torch
            if arr.dtype != torch.uint8 or not arr.is_cuda:
                raise PbhError(f"{name}: device batches must be CUDA uint8 tensors")
            if arr.dim() == 1:
                arr = arr.unsqueeze(0)
            if arr.stride(-1) != 1:
                raise PbhError(f"{name}: planes must be contiguous along the item axis")
            self.arr, self.ptr = arr, arr.data_ptr()
            self.pitch = arr.stride(0) if arr.shape[0] > 1 else max(arr.shape[1], 1)
        else:
            arr = np.asarray(arr)
            if arr.dtype != np.uint8:
                raise PbhError(f"{name}: host batches must be uint8 arrays")
            if arr.ndim == 1:
                arr = arr.reshape(1, -1)
            if arr.shape[1] > 0 and arr.strides[1] != 1:
                if out:      # the library would fill a temporary copy and the caller's array would stay untouched
                    raise PbhError(f"{name}: output planes must be contiguous along the item axis")
                arr = np.ascontiguousarray(arr)
            if out and not arr.flags.writeable:
                raise PbhError(f"{name}: output array is read-only")
            self.arr, self.ptr = arr, arr.ctypes.data
            self.pitch = arr.strides[0] if arr.shape[0] > 1 else max(arr.shape[1], 1)
        if arr.shape[0] != planes:
            raise PbhError(f"{name}: expected {planes} planes, got {arr.shape[0]}")
        if n is not None and arr.shape[1] != n:
            raise PbhError(f"{name}: expected {n} items, got {arr.shape[1]}")
        self.n = arr.shape[1]


class Context:
    """pbh_ctx: SRS::create + Plonk::new + hoisted circuit constants on one CUDA device."""

    def __init__(self, circuit=None, s=2, srs_n=6, omega_pows=4, device=0, algo="table"):
        self.lib = load_library()
        self.circuit = circuit if circuit is not None else pbh_test_circuit()
        self.s, self.srs_n, self.omega_pows, self.device = s, srs_n, omega_pows, device
        h = C.c_void_p()
        rc = self.lib.pbh_ctx_create(C.byref(self.circuit), C.c_uint8(s), C.c_uint32(srs_n), C.c_uint8(omega_pows), int(device),
                                     C.byref(h))
        if rc != 0:
            msg = self.lib.pbh_last_error(None).decode()
            if rc == -2:
                raise ReferencePanic(rc, "setup panics in the reference: " + msg)
            raise PbhError(f"pbh_ctx_create: {ERR.get(rc, rc)}: {msg}")
        self.h = h
        self.set_algo(algo)

    def close(self):
        if getattr(self, "h", None):
            self.lib.pbh_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc != 0:
            raise PbhError(f"{what}: {ERR.get(rc, rc)}: {self.lib.pbh_last_error(self.h).decode()}")

    # ---- context properties ----
    def set_algo(self, algo):
        code = {"arith": ALGO_ARITH, "table": ALGO_TABLE}.get(algo, algo)
        self._check(self.lib.pbh_ctx_set_algo(self.h, int(code)), "pbh_ctx_set_algo")
        self.algo = "table" if code == ALGO_TABLE else "arith"

    def set_option(self, option, value):
        """Tuning switches of include/pbh_b200.h (PBH_OPT_*); results never change."""
        self._check(self.lib.pbh_ctx_set_option(self.h, int(option), int(value)), "pbh_ctx_set_option")

    def sync(self):
        self._check(self.lib.pbh_ctx_sync(self.h), "pbh_ctx_sync")

    @property
    def stream_ptr(self):
        return self.lib.pbh_ctx_stream(self.h)

    def torch_stream(self):
        """The context's compute stream as a torch.cuda.ExternalStream (for CUDA-event timing)."""
        import torch
        return torch.cuda.ExternalStream(self.stream_ptr, device=torch.device("cuda", self.device))

    @property
    def launch_count(self):
        return int(self.lib.pbh_ctx_launch_count(self.h))

    def srs(self):
        n = C.c_uint32()
        g1s = np.zeros(3 * (self.srs_n + 1), dtype=np.uint8)
        g2 = np.zeros(4, dtype=np.uint8)
        self._check(self.lib.pbh_ctx_get_srs(self.h, g1s.ctypes.data_as(u8p), C.c_size_t(self.srs_n + 1), C.byref(n),
                                             g2.ctypes.data_as(u8p)), "pbh_ctx_get_srs")
        return g1s.reshape(-1, 3), g2

    def verifier_constants(self):
        c = np.zeros(24, dtype=np.uint8)
        self._check(self.lib.pbh_ctx_get_verifier_constants(self.h, c.ctypes.data_as(u8p)), "pbh_ctx_get_verifier_constants")
        return c.reshape(8, 3)

    # ---- stream ordering of the device-pointer API ----
    # Kernels run on the context's own (non-blocking) stream.  Around every device-pointer call the context's stream
    # first waits for the caller's current torch stream (inputs are ready) and the caller's stream then waits for the
    # context's stream (outputs are ready), so the calls compose like ordinary torch ops.  Both waits are no-ops when
    # the caller already runs under `with torch.cuda.stream(ctx.torch_stream())`, as bench.py does.
    def _dev_begin(self):
        import torch
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream != self.stream_ptr:
            if not hasattr(self, "_ext"):
                self._ext = self.torch_stream()
            self._ext.wait_stream(cur)
            return cur
        return None

    def _dev_end(self, cur):
        if cur is not None:
            cur.wait_stream(self._ext)

    # ---- allocation helpers ----
    def _empty(self, like_dev, planes, n):
        if like_dev:
            import torch
            return torch.empty((planes, n), dtype=torch.uint8, device=torch.device("cuda", self.device))
        return np.empty((planes, n), dtype=np.uint8)

    # ---- Plonk::prove / Plonk::verify over batches ----
    def prove_batch(self, wit, rand, chal, proof=None, status=None):
        """wit (12,n), rand (9,n), chal (5,n) -> proof (27,n), status (n,).  numpy = host API, torch.cuda = device API."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand"); Ch = _Planes(chal, 5, n, "chal")
        if not (W.dev == R.dev == Ch.dev):
            raise PbhError("all batches must live on the same side (host or device)")
        proof = self._empty(W.dev, 27, n) if proof is None else proof
        status = self._empty(W.dev, 1, n) if status is None else status
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        fn = self.lib.pbh_prove_batch_dev if W.dev else self.lib.pbh_prove_batch
        cur = self._dev_begin() if W.dev else None
        rc = fn(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr), C.c_size_t(R.pitch),
                C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(S.ptr))
        self._dev_end(cur)
        self._check(rc, fn.__name__)
        return P.arr, S.arr.reshape(-1)

    def verify_batch(self, proof, chal, u, result=None, gt=None, want_gt=False):
        """proof (27,n), chal (5,n), u (n,) -> result (n,) of PBH_VR_* [, gt (4,n)]."""
        P = _Planes(proof, 27, name="proof"); n = P.n
        Ch = _Planes(chal, 5, n, "chal"); U = _Planes(u, 1, n, "u")
        if not (P.dev == Ch.dev == U.dev):
            raise PbhError("all batches must live on the same side (host or device)")
        result = self._empty(P.dev, 1, n) if result is None else result
        Rs = _Planes(result, 1, n, "result", out=True)
        G = None
        if want_gt or gt is not None:
            gt = self._empty(P.dev, 4, n) if gt is None else gt
            G = _Planes(gt, 4, n, "gt", out=True)
        fn = self.lib.pbh_verify_batch_dev if P.dev else self.lib.pbh_verify_batch
        cur = self._dev_begin() if P.dev else None
        rc = fn(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch),
                C.c_void_p(U.ptr), C.c_void_p(Rs.ptr), C.c_void_p(G.ptr if G else None), C.c_size_t(G.pitch if G else 0))
        self._dev_end(cur)
        self._check(rc, fn.__name__)
        res = Rs.arr.reshape(-1)
        return (res, G.arr) if G else res

    # ---- asynchronous host-pointer calls on lanes (include/pbh_b200.h) ----
    def prove_batch_async(self, lane, wit, rand, chal, proof, status):
        """Enqueue pbh_prove_batch on `lane` and return; the arrays must stay alive and untouched until lane_sync(lane)."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand"); Ch = _Planes(chal, 5, n, "chal")
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        if W.dev or R.dev or Ch.dev or P.dev or S.dev:
            raise PbhError("the lane API takes host arrays")
        rc = self.lib.pbh_prove_batch_async(self.h, int(lane), C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr),
                                            C.c_size_t(R.pitch), C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch), C.c_void_p(P.ptr),
                                            C.c_size_t(P.pitch), C.c_void_p(S.ptr))
        self._check(rc, "pbh_prove_batch_async")

    def verify_batch_async(self, lane, proof, chal, u, result, gt=None):
        P = _Planes(proof, 27, name="proof"); n = P.n
        Ch = _Planes(chal, 5, n, "chal"); U = _Planes(u, 1, n, "u"); Rs = _Planes(result, 1, n, "result", out=True)
        G = _Planes(gt, 4, n, "gt", out=True) if gt is not None else None
        if P.dev or Ch.dev or U.dev or Rs.dev or (G is not None and G.dev):
            raise PbhError("the lane API takes host arrays")
        rc = self.lib.pbh_verify_batch_async(self.h, int(lane), C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Ch.ptr),
                                             C.c_size_t(Ch.pitch), C.c_void_p(U.ptr), C.c_void_p(Rs.ptr), C.c_void_p(G.ptr if G else None),
                                             C.c_size_t(G.pitch if G else 0))
        self._check(rc, "pbh_verify_batch_async")

    def lane_sync(self, lane):
        self._check(self.lib.pbh_lane_sync(self.h, int(lane)), "pbh_lane_sync")

    @property
    def numa_node(self):
        return int(self.lib.pbh_ctx_numa_node(self.h))

    def host_alloc(self, shape, write_combined=False):
        """uint8 numpy array over page-locked, mapped host memory (pbh_host_alloc): the host-pointer calls run in place
        on it.  The memory lives until host_free(array) or the context closes.  write_combined: pbh_host_alloc_input
        (input buffers only: the host writes, the device reads)."""
        shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        nbytes = max(1, int(np.prod(shape)))
        p = C.c_void_p()
        fn = self.lib.pbh_host_alloc_input if write_combined else self.lib.pbh_host_alloc
        self._check(fn(self.h, C.c_size_t(nbytes), C.byref(p)), "pbh_host_alloc")
        buf = (C.c_uint8 * nbytes).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8, count=int(np.prod(shape))).reshape(shape)
        self._host_ptrs = getattr(self, "_host_ptrs", {})
        self._host_ptrs[arr.ctypes.data] = p.value
        return arr

    def host_free(self, arr):
        p = getattr(self, "_host_ptrs", {}).pop(arr.ctypes.data, None)
        if p is None:
            raise PbhError("not a host_alloc array of this context")
        self._check(self.lib.pbh_host_free(self.h, C.c_void_p(p)), "pbh_host_free")

    def prove_digest_batch(self, wit, rand, chal, proof, status, digest, first_index=0):
        """Device tensors: prove and add the additive digest of the 27 proof planes (== digest(proof, first_index)) in
        the same kernel.  `digest`: int64 tensor of one element."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand"); Ch = _Planes(chal, 5, n, "chal")
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        cur = self._dev_begin()
        rc = self.lib.pbh_prove_digest_batch_dev(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr),
                                                 C.c_size_t(R.pitch), C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch), C.c_void_p(P.ptr),
                                                 C.c_size_t(P.pitch), C.c_void_p(S.ptr), C.c_uint64(first_index),
                                                 C.c_void_p(digest.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_prove_digest_batch_dev")
        return P.arr, S.arr.reshape(-1), digest

    def verify_bitmap_batch(self, proof, chal, u, result, bitmap):
        """Device tensors: verify and pack the verdict bits (== pack_verdicts(result)) in the same kernel."""
        P = _Planes(proof, 27, name="proof"); n = P.n
        Ch = _Planes(chal, 5, n, "chal"); U = _Planes(u, 1, n, "u"); Rs = _Planes(result, 1, n, "result", out=True)
        cur = self._dev_begin()
        rc = self.lib.pbh_verify_bitmap_batch_dev(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Ch.ptr),
                                                  C.c_size_t(Ch.pitch), C.c_void_p(U.ptr), C.c_void_p(Rs.ptr), C.c_void_p(bitmap.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_verify_bitmap_batch_dev")
        return Rs.arr.reshape(-1), bitmap

    def prove_verify_batch(self, wit, rand, chal, u, proof=None, status=None, result=None):
        """Host arrays only: prove, then verify the fresh proofs, with the proofs staying on the device in between."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand"); Ch = _Planes(chal, 5, n, "chal"); U = _Planes(u, 1, n, "u")
        if W.dev or R.dev or Ch.dev or U.dev:
            raise PbhError("prove_verify_batch takes host arrays")
        proof = np.empty((27, n), dtype=np.uint8) if proof is None else proof
        status = np.empty((n,), dtype=np.uint8) if status is None else status
        result = np.empty((n,), dtype=np.uint8) if result is None else result
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True); Rs = _Planes(result, 1, n, "result", out=True)
        rc = self.lib.pbh_prove_verify_batch(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr),
                                             C.c_size_t(R.pitch), C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch), C.c_void_p(U.ptr),
                                             C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(S.ptr), C.c_void_p(Rs.ptr))
        self._check(rc, "pbh_prove_verify_batch")
        return P.arr, S.arr.reshape(-1), Rs.arr.reshape(-1)

    # ---- Fiat-Shamir transcript (include/pbh_b200.h): the challenges and u are derived on the device ----
    def fs_seed(self):
        out = (C.c_uint8 * 32)()
        self._check(self.lib.pbh_ctx_get_fs_seed(self.h, out), "pbh_ctx_get_fs_seed")
        return bytes(out)

    def prove_fs_batch(self, wit, rand, proof=None, status=None, chal=None, want_chal=True):
        """wit (12,n), rand (9,n) -> proof (27,n), status (n,) [, chal (6,n) = alpha beta gamma z v u]."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand")
        if W.dev != R.dev:
            raise PbhError("all batches must live on the same side (host or device)")
        proof = self._empty(W.dev, 27, n) if proof is None else proof
        status = self._empty(W.dev, 1, n) if status is None else status
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        Ch = None
        if want_chal or chal is not None:
            chal = self._empty(W.dev, 6, n) if chal is None else chal
            Ch = _Planes(chal, 6, n, "chal", out=True)
        fn = self.lib.pbh_prove_fs_batch_dev if W.dev else self.lib.pbh_prove_fs_batch
        cur = self._dev_begin() if W.dev else None
        rc = fn(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr), C.c_size_t(R.pitch),
                C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(S.ptr), C.c_void_p(Ch.ptr if Ch else None),
                C.c_size_t(Ch.pitch if Ch else 0))
        self._dev_end(cur)
        self._check(rc, fn.__name__)
        return (P.arr, S.arr.reshape(-1), Ch.arr) if Ch else (P.arr, S.arr.reshape(-1))

    def verify_fs_batch(self, proof, result=None, chal=None, want_chal=True, gt=None, want_gt=False):
        """proof (27,n) -> result (n,) [, chal (6,n)] [, gt (4,n)]."""
        P = _Planes(proof, 27, name="proof"); n = P.n
        result = self._empty(P.dev, 1, n) if result is None else result
        Rs = _Planes(result, 1, n, "result", out=True)
        Ch = G = None
        if want_chal or chal is not None:
            chal = self._empty(P.dev, 6, n) if chal is None else chal
            Ch = _Planes(chal, 6, n, "chal", out=True)
        if want_gt or gt is not None:
            gt = self._empty(P.dev, 4, n) if gt is None else gt
            G = _Planes(gt, 4, n, "gt", out=True)
        fn = self.lib.pbh_verify_fs_batch_dev if P.dev else self.lib.pbh_verify_fs_batch
        cur = self._dev_begin() if P.dev else None
        rc = fn(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Rs.ptr), C.c_void_p(Ch.ptr if Ch else None),
                C.c_size_t(Ch.pitch if Ch else 0), C.c_void_p(G.ptr if G else None), C.c_size_t(G.pitch if G else 0))
        self._dev_end(cur)
        self._check(rc, fn.__name__)
        out = [Rs.arr.reshape(-1)]
        if Ch: out.append(Ch.arr)
        if G: out.append(G.arr)
        return out[0] if len(out) == 1 else tuple(out)

    def prove_fs_digest_batch(self, wit, rand, proof, status, digest, first_index=0, chal=None):
        """Device tensors: prove_fs_batch and the additive digest of the 27 proof planes (== digest(proof, first_index)), fused
        into the FP32 provers.  `digest`: int64 tensor of one element, overwritten.  chal (6,n): optional derived challenges."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand")
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        Ch = _Planes(chal, 6, n, "chal", out=True) if chal is not None else None
        if not (W.dev and R.dev and P.dev and S.dev and (Ch is None or Ch.dev)):
            raise PbhError("prove_fs_digest_batch takes CUDA tensors")
        cur = self._dev_begin()
        rc = self.lib.pbh_prove_fs_digest_batch_dev(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr),
                                                    C.c_size_t(R.pitch), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(S.ptr),
                                                    C.c_void_p(Ch.ptr if Ch else None), C.c_size_t(Ch.pitch if Ch else 0),
                                                    C.c_uint64(first_index), C.c_void_p(digest.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_prove_fs_digest_batch_dev")
        return P.arr, S.arr.reshape(-1), digest

    def verify_fs_bitmap_batch(self, proof, result, bitmap):
        """Device tensors: verify_fs_batch and the packed verdict bits (== pack_verdicts(result)), fused when `bitmap` is
        4-byte aligned."""
        P = _Planes(proof, 27, name="proof"); n = P.n
        Rs = _Planes(result, 1, n, "result", out=True)
        if not (P.dev and Rs.dev):
            raise PbhError("verify_fs_bitmap_batch takes CUDA tensors")
        cur = self._dev_begin()
        rc = self.lib.pbh_verify_fs_bitmap_batch_dev(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Rs.ptr),
                                                     C.c_void_p(bitmap.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_verify_fs_bitmap_batch_dev")
        return Rs.arr.reshape(-1), bitmap

    # ---- record (array-of-structs) wire format ----
    def prove_records(self, records):
        """records: numpy array of WITNESS_RECORD (host) -> numpy array of PROOF_RECORD."""
        rec = np.ascontiguousarray(records, dtype=WITNESS_RECORD)
        out = np.zeros(rec.shape[0], dtype=PROOF_RECORD)
        rc = self.lib.pbh_prove_records(self.h, C.c_size_t(rec.shape[0]), C.c_void_p(rec.ctypes.data), C.c_void_p(out.ctypes.data))
        self._check(rc, "pbh_prove_records")
        return out

    def verify_records(self, proofs, params):
        prf = np.ascontiguousarray(proofs, dtype=PROOF_RECORD); par = np.ascontiguousarray(params, dtype=WITNESS_RECORD)
        if prf.shape[0] != par.shape[0]:
            raise PbhError("proofs and params must have the same length")
        res = np.zeros(prf.shape[0], dtype=np.uint8)
        rc = self.lib.pbh_verify_records(self.h, C.c_size_t(prf.shape[0]), C.c_void_p(prf.ctypes.data), C.c_void_p(par.ctypes.data),
                                         C.c_void_p(res.ctypes.data))
        self._check(rc, "pbh_verify_records")
        return res

    # ---- peer windows: the shard summaries stored into every peer's buffer by the kernels that produce them ----
    def window_create(self, bytes_per_rank, rank, world):
        """-> (torch uint8 tensor of shape (world, bytes_per_rank) over this rank's window, 64-byte IPC handle as numpy uint8).
        Rank r's region is row r of EVERY rank's tensor; summaries written into the own row (the `digest` of
        prove_digest_batch, the `bitmap` of verify_bitmap_batch) appear in the same place of every attached peer."""
        import torch
        base = C.c_void_p()
        handle = np.zeros(64, dtype=np.uint8)
        self._check(self.lib.pbh_window_create(self.h, C.c_size_t(bytes_per_rank), int(rank), int(world), C.byref(base),
                                               C.c_void_p(handle.ctypes.data)), "pbh_window_create")

        class _Dev:   # CUDA array interface over library-owned device memory (lives until window_destroy / close)
            __cuda_array_interface__ = {"shape": (int(world) * int(bytes_per_rank),), "typestr": "|u1", "data": (int(base.value), False), "version": 3}
        with torch.cuda.device(self.device):
            t = torch.as_tensor(_Dev(), device=torch.device("cuda", self.device))
        self._window_base = int(base.value)
        return t.view(int(world), int(bytes_per_rank)), handle

    def window_attach(self, handles):
        """handles: (world, 64) uint8 array, row r = rank r's IPC handle (other processes)."""
        hs = np.ascontiguousarray(handles, dtype=np.uint8)
        self._check(self.lib.pbh_window_attach(self.h, C.c_void_p(hs.ctypes.data)), "pbh_window_attach")

    def window_attach_ptrs(self, bases):
        """bases: one device address per rank (peers of this process; the own entry is ignored)."""
        arr = (C.c_void_p * len(bases))(*[C.c_void_p(int(b)) for b in bases])
        self._check(self.lib.pbh_window_attach_ptrs(self.h, arr), "pbh_window_attach_ptrs")

    def window_share(self, other):
        self._check(self.lib.pbh_window_share(self.h, other.h), "pbh_window_share")

    def window_destroy(self):
        self._check(self.lib.pbh_window_destroy(self.h), "pbh_window_destroy")

    # ---- packed wire format (16-byte prover inputs, 12-byte proofs, 4-byte challenge words) ----
    @staticmethod
    def _packed(a, dtype, name, out=False):
        a = np.asarray(a)
        if a.dtype != dtype or a.ndim != 1 or not a.flags.c_contiguous or (out and not a.flags.writeable):
            raise PbhError(f"{name}: expected a contiguous 1-D array of {dtype}")
        return a

    def prove_packed(self, packed_in, out=None):
        """PACKED_WITNESS array (host) -> PACKED_PROOF array: pack(pbh_prove_batch(unpack(in)))."""
        pin = self._packed(packed_in, PACKED_WITNESS, "packed_in"); n = pin.shape[0]
        out = np.zeros(n, dtype=PACKED_PROOF) if out is None else self._packed(out, PACKED_PROOF, "out", True)
        self._check(self.lib.pbh_prove_packed(self.h, C.c_size_t(n), C.c_void_p(pin.ctypes.data), C.c_void_p(out.ctypes.data)), "pbh_prove_packed")
        return out

    def verify_packed(self, proofs, chal_u, result=None):
        prf = self._packed(proofs, PACKED_PROOF, "proofs"); n = prf.shape[0]
        cu = self._packed(chal_u, np.dtype("<u4"), "chal_u")
        if cu.shape[0] != n:
            raise PbhError("proofs and chal_u must have the same length")
        res = np.zeros(n, dtype=np.uint8) if result is None else self._packed(result, np.dtype(np.uint8), "result", True)
        self._check(self.lib.pbh_verify_packed(self.h, C.c_size_t(n), C.c_void_p(prf.ctypes.data), C.c_void_p(cu.ctypes.data),
                                               C.c_void_p(res.ctypes.data)), "pbh_verify_packed")
        return res

    def prove_verify_packed(self, packed_in, out=None, result=None):
        pin = self._packed(packed_in, PACKED_WITNESS, "packed_in"); n = pin.shape[0]
        out = np.zeros(n, dtype=PACKED_PROOF) if out is None else self._packed(out, PACKED_PROOF, "out", True)
        res = np.zeros(n, dtype=np.uint8) if result is None else self._packed(result, np.dtype(np.uint8), "result", True)
        self._check(self.lib.pbh_prove_verify_packed(self.h, C.c_size_t(n), C.c_void_p(pin.ctypes.data), C.c_void_p(out.ctypes.data),
                                                     C.c_void_p(res.ctypes.data)), "pbh_prove_verify_packed")
        return out, res

    def prove_packed_async(self, lane, packed_in, out):
        """Enqueue pbh_prove_packed on `lane`; the arrays must stay alive and untouched until lane_sync(lane)."""
        pin = self._packed(packed_in, PACKED_WITNESS, "packed_in"); o = self._packed(out, PACKED_PROOF, "out", True)
        if o.shape[0] != pin.shape[0]:
            raise PbhError("packed_in and out must have the same length")
        self._check(self.lib.pbh_prove_packed_async(self.h, int(lane), C.c_size_t(pin.shape[0]), C.c_void_p(pin.ctypes.data),
                                                    C.c_void_p(o.ctypes.data)), "pbh_prove_packed_async")

    def verify_packed_async(self, lane, proofs, chal_u, result):
        prf = self._packed(proofs, PACKED_PROOF, "proofs"); cu = self._packed(chal_u, np.dtype("<u4"), "chal_u")
        res = self._packed(result, np.dtype(np.uint8), "result", True)
        if cu.shape[0] != prf.shape[0] or res.shape[0] != prf.shape[0]:
            raise PbhError("proofs, chal_u and result must have the same length")
        self._check(self.lib.pbh_verify_packed_async(self.h, int(lane), C.c_size_t(prf.shape[0]), C.c_void_p(prf.ctypes.data),
                                                     C.c_void_p(cu.ctypes.data), C.c_void_p(res.ctypes.data)), "pbh_verify_packed_async")

    def prove_verify_packed_async(self, lane, packed_in, out, result):
        pin = self._packed(packed_in, PACKED_WITNESS, "packed_in"); o = self._packed(out, PACKED_PROOF, "out", True)
        res = self._packed(result, np.dtype(np.uint8), "result", True)
        if o.shape[0] != pin.shape[0] or res.shape[0] != pin.shape[0]:
            raise PbhError("packed_in, out and result must have the same length")
        self._check(self.lib.pbh_prove_verify_packed_async(self.h, int(lane), C.c_size_t(pin.shape[0]), C.c_void_p(pin.ctypes.data),
                                                           C.c_void_p(o.ctypes.data), C.c_void_p(res.ctypes.data)), "pbh_prove_verify_packed_async")

    # ---- Fiat-Shamir over packed records (12-byte prover inputs, 12-byte proofs, optional 4-byte challenge words) ----
    # numpy arrays select the host-pointer calls; CUDA tensors (contiguous, any dtype, viewed as bytes) select the `_dev` calls,
    # whose outputs are uint8 tensors of 12 (proofs) / 4 (challenge words) / 1 (results) bytes per item.
    def _dev_records(self, t, itemsize, name, n=None):
        if not t.is_cuda or not t.is_contiguous():
            raise PbhError(f"{name}: device records must be a contiguous CUDA tensor")
        nbytes = t.numel() * t.element_size()
        if nbytes % itemsize or (n is not None and nbytes != n * itemsize):
            raise PbhError(f"{name}: expected {'n' if n is None else n} records of {itemsize} bytes, got {nbytes} bytes")
        return t, nbytes // itemsize

    def _dev_bytes(self, n, itemsize):
        import torch
        return torch.empty((n * itemsize,), dtype=torch.uint8, device=torch.device("cuda", self.device))

    def prove_fs_packed(self, packed_in, out=None, chal_u=None, want_chal_u=True):
        """PACKED_FS_WITNESS records -> PACKED_PROOF records [, challenge words alpha beta gamma z v u]:
        pack(pbh_prove_fs_batch(unpack(in))).  numpy = host call, torch.cuda = device call."""
        if _is_torch(packed_in):
            pin, n = self._dev_records(packed_in, 12, "packed_in")
            out = self._dev_bytes(n, 12) if out is None else self._dev_records(out, 12, "out", n)[0]
            if want_chal_u or chal_u is not None:
                chal_u = self._dev_bytes(n, 4) if chal_u is None else self._dev_records(chal_u, 4, "chal_u", n)[0]
            cur = self._dev_begin()
            rc = self.lib.pbh_prove_fs_packed_dev(self.h, C.c_size_t(n), C.c_void_p(pin.data_ptr()), C.c_void_p(out.data_ptr()),
                                                  C.c_void_p(chal_u.data_ptr() if chal_u is not None else None))
            self._dev_end(cur)
            self._check(rc, "pbh_prove_fs_packed_dev")
        else:
            pin = self._packed(packed_in, PACKED_FS_WITNESS, "packed_in"); n = pin.shape[0]
            out = np.zeros(n, dtype=PACKED_PROOF) if out is None else self._packed(out, PACKED_PROOF, "out", True)
            if want_chal_u or chal_u is not None:
                chal_u = np.zeros(n, dtype="<u4") if chal_u is None else self._packed(chal_u, np.dtype("<u4"), "chal_u", True)
            if out.shape[0] != n or (chal_u is not None and chal_u.shape[0] != n):
                raise PbhError("packed_in, out and chal_u must have the same length")
            self._check(self.lib.pbh_prove_fs_packed(self.h, C.c_size_t(n), C.c_void_p(pin.ctypes.data), C.c_void_p(out.ctypes.data),
                                                     C.c_void_p(chal_u.ctypes.data if chal_u is not None else None)), "pbh_prove_fs_packed")
        return (out, chal_u) if chal_u is not None else out

    def verify_fs_packed(self, proofs, result=None):
        """PACKED_PROOF records -> result bytes (PBH_VR_*): pbh_verify_fs_batch(unpack(proofs)).  numpy = host, torch.cuda = device."""
        if _is_torch(proofs):
            prf, n = self._dev_records(proofs, 12, "proofs")
            result = self._dev_bytes(n, 1) if result is None else self._dev_records(result, 1, "result", n)[0]
            cur = self._dev_begin()
            rc = self.lib.pbh_verify_fs_packed_dev(self.h, C.c_size_t(n), C.c_void_p(prf.data_ptr()), C.c_void_p(result.data_ptr()))
            self._dev_end(cur)
            self._check(rc, "pbh_verify_fs_packed_dev")
            return result
        prf = self._packed(proofs, PACKED_PROOF, "proofs"); n = prf.shape[0]
        res = np.zeros(n, dtype=np.uint8) if result is None else self._packed(result, np.dtype(np.uint8), "result", True)
        if res.shape[0] != n:
            raise PbhError("proofs and result must have the same length")
        self._check(self.lib.pbh_verify_fs_packed(self.h, C.c_size_t(n), C.c_void_p(prf.ctypes.data), C.c_void_p(res.ctypes.data)),
                    "pbh_verify_fs_packed")
        return res

    def prove_fs_packed_async(self, lane, packed_in, out, chal_u=None):
        """Enqueue pbh_prove_fs_packed on `lane`; the arrays must stay alive and untouched until lane_sync(lane)."""
        pin = self._packed(packed_in, PACKED_FS_WITNESS, "packed_in"); o = self._packed(out, PACKED_PROOF, "out", True)
        cu = self._packed(chal_u, np.dtype("<u4"), "chal_u", True) if chal_u is not None else None
        if o.shape[0] != pin.shape[0] or (cu is not None and cu.shape[0] != pin.shape[0]):
            raise PbhError("packed_in, out and chal_u must have the same length")
        self._check(self.lib.pbh_prove_fs_packed_async(self.h, int(lane), C.c_size_t(pin.shape[0]), C.c_void_p(pin.ctypes.data),
                                                       C.c_void_p(o.ctypes.data), C.c_void_p(cu.ctypes.data if cu is not None else None)),
                    "pbh_prove_fs_packed_async")

    def verify_fs_packed_async(self, lane, proofs, result):
        prf = self._packed(proofs, PACKED_PROOF, "proofs"); res = self._packed(result, np.dtype(np.uint8), "result", True)
        if res.shape[0] != prf.shape[0]:
            raise PbhError("proofs and result must have the same length")
        self._check(self.lib.pbh_verify_fs_packed_async(self.h, int(lane), C.c_size_t(prf.shape[0]), C.c_void_p(prf.ctypes.data),
                                                        C.c_void_p(res.ctypes.data)), "pbh_verify_fs_packed_async")

    def host_alloc_as(self, n, dtype, write_combined=False):
        """host_alloc viewed as n records of `dtype` (page-locked memory for the packed lane calls)."""
        dtype = np.dtype(dtype)
        raw = self.host_alloc(max(1, int(n)) * dtype.itemsize, write_combined=write_combined)
        arr = raw[:int(n) * dtype.itemsize].view(dtype)
        self._host_ptrs[arr.ctypes.data] = self._host_ptrs[raw.ctypes.data]
        return arr

    def unpack_witness_dev(self, packed_dev, n):
        """Device conversion: torch uint8 tensor holding n PACKED_WITNESS records -> (wit, rand, chal, u) device planes."""
        import torch
        wit, rand, chal = (torch.empty((k, n), dtype=torch.uint8, device=packed_dev.device) for k in (12, 9, 5))
        u = torch.empty((n,), dtype=torch.uint8, device=packed_dev.device)
        cur = self._dev_begin()
        rc = self.lib.pbh_unpack_witness_dev(self.h, C.c_size_t(n), C.c_void_p(packed_dev.data_ptr()), C.c_void_p(wit.data_ptr()), C.c_size_t(n),
                                             C.c_void_p(rand.data_ptr()), C.c_size_t(n), C.c_void_p(chal.data_ptr()), C.c_size_t(n), C.c_void_p(u.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_unpack_witness_dev")
        return wit, rand, chal, u

    def pack_proof_dev(self, proof, status):
        """Device conversion: (27, n) proof planes + status -> torch uint8 tensor of n 12-byte PACKED_PROOF records."""
        import torch
        P = _Planes(proof, 27, name="proof"); n = P.n
        out = torch.empty((n * 12,), dtype=torch.uint8, device=proof.device)
        cur = self._dev_begin()
        rc = self.lib.pbh_pack_proof_dev(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch),
                                         C.c_void_p(status.data_ptr() if status is not None else None), C.c_void_p(out.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_pack_proof_dev")
        return out

    def unpack_proof_dev(self, packed_dev, chal_u_dev, n):
        """Device conversion: packed proofs (+ challenge words) -> (proof planes, status, chal planes, u)."""
        import torch
        dev = packed_dev.device
        proof = torch.empty((27, n), dtype=torch.uint8, device=dev); status = torch.empty((n,), dtype=torch.uint8, device=dev)
        chal = torch.empty((5, n), dtype=torch.uint8, device=dev); u = torch.empty((n,), dtype=torch.uint8, device=dev)
        cur = self._dev_begin()
        rc = self.lib.pbh_unpack_proof_dev(self.h, C.c_size_t(n), C.c_void_p(packed_dev.data_ptr()),
                                           C.c_void_p(chal_u_dev.data_ptr() if chal_u_dev is not None else None), C.c_void_p(proof.data_ptr()),
                                           C.c_size_t(n), C.c_void_p(status.data_ptr()), C.c_void_p(chal.data_ptr()), C.c_size_t(n), C.c_void_p(u.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_unpack_proof_dev")
        return proof, status, chal, u

    # ---- sweep kernels ----
    def _sweep(self, fn, arr, pin, pout, *pre):
        A = _Planes(arr, pin, name="in")
        out = self._empty(A.dev, pout, A.n)
        O = _Planes(out, pout, A.n, "out")
        cur = self._dev_begin() if A.dev else None
        rc = fn(self.h, *pre, C.c_size_t(A.n), C.c_void_p(A.ptr), C.c_size_t(A.pitch), C.c_void_p(O.ptr), C.c_size_t(O.pitch),
                int(A.dev))
        self._dev_end(cur)
        self._check(rc, fn.__name__)
        return O.arr

    def ntt4_batch(self, coeffs): return self._sweep(self.lib.pbh_ntt4_batch, coeffs, 4, 4)
    def intt4_batch(self, evals): return self._sweep(self.lib.pbh_intt4_batch, evals, 4, 4)

    def _coset(self, fn, arr, k):
        A = _Planes(arr, 4, name="in")
        out = self._empty(A.dev, 4, A.n)
        O = _Planes(out, 4, A.n, "out")
        cur = self._dev_begin() if A.dev else None
        rc = fn(self.h, C.c_size_t(A.n), C.c_uint32(k), C.c_void_p(A.ptr), C.c_size_t(A.pitch), C.c_void_p(O.ptr), C.c_size_t(O.pitch), int(A.dev))
        self._dev_end(cur)
        self._check(rc, fn.__name__)
        return O.arr

    def coset_ntt4_batch(self, coeffs, k):
        """evals[i] = p(k 4^i): the coset k H of src/plonk.rs:136-139 (k = 2: K1, k = 3: K2, k = 1: H)."""
        return self._coset(self.lib.pbh_coset_ntt4_batch, coeffs, k)

    def coset_intt4_batch(self, evals, k):
        return self._coset(self.lib.pbh_coset_intt4_batch, evals, k)
    def g1_smul_batch(self, arr): return self._sweep(self.lib.pbh_g1_smul_batch, arr, 4, 3)
    def g1_add_batch(self, arr): return self._sweep(self.lib.pbh_g1_add_batch, arr, 6, 3)
    def kzg_commit_batch(self, arr): return self._sweep(self.lib.pbh_kzg_commit_batch, arr, 7, 3)
    def pairing_batch(self, arr): return self._sweep(self.lib.pbh_pairing_batch, arr, 5, 2)
    def gt_mul_batch(self, arr): return self._sweep(self.lib.pbh_gt_mul_batch, arr, 4, 2)
    def gt_pow600_batch(self, arr): return self._sweep(self.lib.pbh_gt_pow600_batch, arr, 2, 2)

    def poly_divrem_batch(self, num, den):
        """num (ln, n), den (ld, n) host arrays -> q (ln, n), r (ld, n), status (n,): src/poly.rs:230-247 for any divisor."""
        N = _Planes(num, np.shape(num)[0], name="num"); D = _Planes(den, np.shape(den)[0], N.n, "den")
        ln, ld = N.arr.shape[0], D.arr.shape[0]
        q = np.empty((ln, N.n), np.uint8); r = np.empty((ld, N.n), np.uint8); st = np.empty((N.n,), np.uint8)
        Q = _Planes(q, ln, N.n, "q", out=True); R = _Planes(r, ld, N.n, "r", out=True)
        rc = self.lib.pbh_poly_divrem_batch(self.h, C.c_size_t(N.n), C.c_uint32(ln), C.c_uint32(ld), C.c_void_p(N.ptr), C.c_size_t(N.pitch),
                                            C.c_void_p(D.ptr), C.c_size_t(D.pitch), C.c_void_p(Q.ptr), C.c_size_t(Q.pitch), C.c_void_p(R.ptr),
                                            C.c_size_t(R.pitch), C.c_void_p(st.ctypes.data), 0)
        self._check(rc, "pbh_poly_divrem_batch")
        return q, r, st

    def poly_addsub_ragged_batch(self, a, b, subtract=False):
        """a (la, n), b (lb, n) host arrays -> (max(la, lb), n): the reference's += / -= for different lengths (Q1 included)."""
        A = _Planes(a, np.shape(a)[0], name="a"); B = _Planes(b, np.shape(b)[0], A.n, "b")
        la, lb = A.arr.shape[0], B.arr.shape[0]
        out = np.empty((max(la, lb), A.n), np.uint8); O = _Planes(out, max(la, lb), A.n, "out", out=True)
        rc = self.lib.pbh_poly_addsub_ragged_batch(self.h, C.c_size_t(A.n), C.c_uint32(la), C.c_uint32(lb), int(subtract), C.c_void_p(A.ptr),
                                                   C.c_size_t(A.pitch), C.c_void_p(B.ptr), C.c_size_t(B.pitch), C.c_void_p(O.ptr), C.c_size_t(O.pitch), 0)
        self._check(rc, "pbh_poly_addsub_ragged_batch")
        return out

    def poly_mul_batch(self, a, b):
        A = _Planes(a, np.shape(a)[0] if not _is_torch(a) else a.shape[0], name="a")
        B = _Planes(b, np.shape(b)[0] if not _is_torch(b) else b.shape[0], A.n, "b")
        la, lb = A.arr.shape[0], B.arr.shape[0]
        out = self._empty(A.dev, la + lb - 1, A.n); O = _Planes(out, la + lb - 1, A.n, "out")
        cur = self._dev_begin() if A.dev else None
        rc = self.lib.pbh_poly_mul_batch(self.h, C.c_size_t(A.n), C.c_uint32(la), C.c_uint32(lb), C.c_void_p(A.ptr),
                                         C.c_size_t(A.pitch), C.c_void_p(B.ptr), C.c_size_t(B.pitch), C.c_void_p(O.ptr),
                                         C.c_size_t(O.pitch), int(A.dev))
        self._dev_end(cur)
        self._check(rc, "pbh_poly_mul_batch")
        return O.arr

    def poly_add_batch(self, a, b, subtract=False):
        ln = a.shape[0]
        A = _Planes(a, ln, name="a"); B = _Planes(b, ln, A.n, "b")
        out = self._empty(A.dev, ln, A.n); O = _Planes(out, ln, A.n, "out")
        cur = self._dev_begin() if A.dev else None
        rc = self.lib.pbh_poly_add_batch(self.h, C.c_size_t(A.n), C.c_uint32(ln), int(subtract), C.c_void_p(A.ptr),
                                         C.c_size_t(A.pitch), C.c_void_p(B.ptr), C.c_size_t(B.pitch), C.c_void_p(O.ptr),
                                         C.c_size_t(O.pitch), int(A.dev))
        self._dev_end(cur)
        self._check(rc, "pbh_poly_add_batch")
        return O.arr

    def poly_div_zh_batch(self, p):
        P = _Planes(p, 22, name="p")
        q = self._empty(P.dev, 18, P.n); r = self._empty(P.dev, 4, P.n)
        Q = _Planes(q, 18, P.n, "q"); R = _Planes(r, 4, P.n, "r")
        cur = self._dev_begin() if P.dev else None
        rc = self.lib.pbh_poly_div_zh_batch(self.h, C.c_size_t(P.n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Q.ptr),
                                            C.c_size_t(Q.pitch), C.c_void_p(R.ptr), C.c_size_t(R.pitch), int(P.dev))
        self._dev_end(cur)
        self._check(rc, "pbh_poly_div_zh_batch")
        return Q.arr, R.arr

    def ntt_generic_batch(self, values, modulus, omega, inverse=False):
        """values: (size, n) uint16 numpy array (host) -> (size, n) uint16.  CooleyTurkey::fft / fft_inv, src/fft.rs:66-78."""
        v = np.ascontiguousarray(values, dtype=np.uint16)
        size, n = v.shape
        out = np.empty_like(v)
        rc = self.lib.pbh_ntt_generic_batch(self.h, C.c_size_t(n), C.c_uint32(modulus), C.c_uint32(omega), C.c_uint32(size),
                                            int(inverse), v.ctypes.data_as(u16p), C.c_size_t(n), out.ctypes.data_as(u16p),
                                            C.c_size_t(n), 0)
        self._check(rc, "pbh_ntt_generic_batch")
        return out

    def mul_ntt_batch(self, a, b, modulus, omega):
        """a (la, n), b (lb, n) uint16 numpy arrays (host) -> (la + lb, n): mul_ntt over CooleyTurkey, src/fft.rs:109-132."""
        a = np.ascontiguousarray(a, dtype=np.uint16); b = np.ascontiguousarray(b, dtype=np.uint16)
        la, n = a.shape; lb = b.shape[0]
        out = np.empty((la + lb, n), dtype=np.uint16)
        rc = self.lib.pbh_mul_ntt_batch(self.h, C.c_size_t(n), C.c_uint32(modulus), C.c_uint32(omega), C.c_uint32(la), C.c_uint32(lb),
                                        a.ctypes.data_as(u16p), C.c_size_t(n), b.ctypes.data_as(u16p), C.c_size_t(n),
                                        out.ctypes.data_as(u16p), C.c_size_t(n), 0)
        self._check(rc, "pbh_mul_ntt_batch")
        return out

    def _poly_unary(self, fn, arr, pout):
        A = _Planes(arr, np.shape(arr)[0] if not _is_torch(arr) else arr.shape[0], name="in")
        ln = A.arr.shape[0] - 1
        out = self._empty(A.dev, pout(ln), A.n)
        O = _Planes(out, pout(ln), A.n, "out")
        cur = self._dev_begin() if A.dev else None
        args = [self.h, C.c_size_t(A.n), C.c_uint32(ln), C.c_void_p(A.ptr), C.c_size_t(A.pitch), C.c_void_p(O.ptr)]
        if fn is not self.lib.pbh_poly_eval_batch:
            args.append(C.c_size_t(O.pitch))
        rc = fn(*args, int(A.dev))
        self._dev_end(cur)
        self._check(rc, "poly sweep")
        return O.arr

    def poly_scale_batch(self, arr):
        """len coefficient planes + the scalar plane -> len planes (src/poly.rs:220-228)."""
        return self._poly_unary(self.lib.pbh_poly_scale_batch, arr, lambda ln: ln)

    def poly_eval_batch(self, arr):
        """len coefficient planes + the point plane -> (n,) (src/poly.rs:71-79)."""
        return self._poly_unary(self.lib.pbh_poly_eval_batch, arr, lambda ln: 1).reshape(-1)

    def poly_div_linear_batch(self, arr):
        """len coefficient planes + the plane c -> len - 1 quotient planes of p / (x - c), then the remainder (src/poly.rs:230-247)."""
        return self._poly_unary(self.lib.pbh_poly_div_linear_batch, arr, lambda ln: ln)

    # ---- device-side helpers (torch) ----
    def generate_inputs(self, n, first_index=0, seed=0xB200, dist=DIST_FULLPATH, want_attempt=False):
        """Synthetic batch on the device (SURVEY.md §8d): returns torch uint8 tensors wit, rand, chal, u[, attempt]."""
        import torch
        dev = torch.device("cuda", self.device)
        wit = torch.empty((12, n), dtype=torch.uint8, device=dev); rand = torch.empty((9, n), dtype=torch.uint8, device=dev)
        chal = torch.empty((5, n), dtype=torch.uint8, device=dev); u = torch.empty((n,), dtype=torch.uint8, device=dev)
        att = torch.empty((n,), dtype=torch.uint8, device=dev) if want_attempt else None
        cur = self._dev_begin()
        rc = self.lib.pbh_generate_inputs_dev(self.h, C.c_size_t(n), C.c_uint64(first_index), C.c_uint64(seed), int(dist),
                                              C.c_void_p(wit.data_ptr()), C.c_size_t(n), C.c_void_p(rand.data_ptr()), C.c_size_t(n),
                                              C.c_void_p(chal.data_ptr()), C.c_size_t(n), C.c_void_p(u.data_ptr()),
                                              C.c_void_p(att.data_ptr() if want_attempt else None))
        self._dev_end(cur)
        self._check(rc, "pbh_generate_inputs_dev")
        return (wit, rand, chal, u, att) if want_attempt else (wit, rand, chal, u)

    def pack_verdicts(self, result, out=None):
        import torch
        n = result.numel()
        if out is None:
            out = torch.empty(((n + 7) // 8,), dtype=torch.uint8, device=result.device)
        cur = self._dev_begin()
        rc = self.lib.pbh_pack_verdicts_dev(self.h, C.c_size_t(n), C.c_void_p(result.data_ptr()), C.c_void_p(out.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_pack_verdicts_dev")
        return out

    def digest(self, data, first_index=0, out=None):
        """64-bit additive digest of a (planes, n) device batch; digests of disjoint shards sum to the whole batch's.
        `out`: optional int64 tensor of one element (8-byte aligned)."""
        import torch
        D = _Planes(data, data.shape[0] if data.dim() > 1 else 1, name="data")
        if out is None:
            out = torch.empty((1,), dtype=torch.int64, device=D.arr.device)     # zeroed by the library on its own stream
        cur = self._dev_begin()
        rc = self.lib.pbh_digest_dev(self.h, C.c_size_t(D.n), C.c_uint64(first_index), C.c_uint32(D.arr.shape[0]), C.c_void_p(D.ptr),
                                     C.c_size_t(D.pitch), C.c_void_p(out.data_ptr()))
        self._dev_end(cur)
        self._check(rc, "pbh_digest_dev")
        return out

    def measure_int32_peak(self, which=0):
        v = C.c_double()
        self._check(self.lib.pbh_measure_int32_peak(self.h, int(which), C.byref(v)), "pbh_measure_int32_peak")
        return v.value


class MultiContext:
    """pbh_multi: one process, several devices (include/pbh_b200.h "multi-device").  Host arrays only."""

    def __init__(self, devices, circuit=None, s=2, srs_n=6, omega_pows=4, algo="table"):
        self.lib = load_library()
        self.circuit = circuit if circuit is not None else pbh_test_circuit()
        devices = list(range(devices)) if isinstance(devices, int) else list(devices)
        arr = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self.lib.pbh_multi_create(C.byref(self.circuit), C.c_uint8(s), C.c_uint32(srs_n), C.c_uint8(omega_pows), arr, len(devices), C.byref(h))
        if rc != 0:
            raise PbhError(f"pbh_multi_create: {ERR.get(rc, rc)}: {self.lib.pbh_multi_last_error(None).decode()}")
        self.h, self.devices = h, devices
        self._check(self.lib.pbh_multi_set_algo(self.h, {"arith": ALGO_ARITH, "table": ALGO_TABLE}[algo]), "pbh_multi_set_algo")

    def _check(self, rc, what):
        if rc != 0:
            raise PbhError(f"{what}: {ERR.get(rc, rc)}: {self.lib.pbh_multi_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.pbh_multi_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_count(self):
        return int(self.lib.pbh_multi_device_count(self.h))

    def prove_batch(self, wit, rand, chal):
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand"); Ch = _Planes(chal, 5, n, "chal")
        proof = np.empty((27, n), np.uint8); status = np.empty((n,), np.uint8)
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        rc = self.lib.pbh_multi_prove_batch(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr), C.c_size_t(R.pitch),
                                            C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(S.ptr))
        self._check(rc, "pbh_multi_prove_batch")
        return proof, status

    def verify_batch(self, proof, chal, u, want_gt=False):
        P = _Planes(proof, 27, name="proof"); n = P.n
        Ch = _Planes(chal, 5, n, "chal"); U = _Planes(u, 1, n, "u")
        result = np.empty((n,), np.uint8); gt = np.empty((4, n), np.uint8) if want_gt else None
        Rs = _Planes(result, 1, n, "result", out=True); G = _Planes(gt, 4, n, "gt", out=True) if want_gt else None
        rc = self.lib.pbh_multi_verify_batch(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Ch.ptr), C.c_size_t(Ch.pitch),
                                             C.c_void_p(U.ptr), C.c_void_p(Rs.ptr), C.c_void_p(G.ptr if G else None), C.c_size_t(G.pitch if G else 0))
        self._check(rc, "pbh_multi_verify_batch")
        return (result, gt) if want_gt else result

    def prove_packed(self, packed_in):
        pin = Context._packed(packed_in, PACKED_WITNESS, "packed_in"); n = pin.shape[0]
        out = np.zeros(n, dtype=PACKED_PROOF)
        self._check(self.lib.pbh_multi_prove_packed(self.h, C.c_size_t(n), C.c_void_p(pin.ctypes.data), C.c_void_p(out.ctypes.data)), "pbh_multi_prove_packed")
        return out

    def verify_packed(self, proofs, chal_u):
        prf = Context._packed(proofs, PACKED_PROOF, "proofs"); cu = Context._packed(chal_u, np.dtype("<u4"), "chal_u")
        res = np.zeros(prf.shape[0], dtype=np.uint8)
        self._check(self.lib.pbh_multi_verify_packed(self.h, C.c_size_t(prf.shape[0]), C.c_void_p(prf.ctypes.data), C.c_void_p(cu.ctypes.data),
                                                     C.c_void_p(res.ctypes.data)), "pbh_multi_verify_packed")
        return res

    def prove_verify_sharded(self, n_total, first_index=0, seed=0xB200, dist=DIST_FULLPATH):
        """-> dict(bitmap uint8[ceil(n/8)], digests uint64[n_dev], total_digest int, accepted int, ms float)."""
        return self._sharded(self.lib.pbh_multi_prove_verify_sharded, n_total, first_index, seed, dist)

    def prove_verify_fs_sharded(self, n_total, first_index=0, seed=0xB200, dist=DIST_FULLPATH):
        """prove_verify_sharded with the Fiat-Shamir transcript (the generated challenges are not used); same dict."""
        return self._sharded(self.lib.pbh_multi_prove_verify_fs_sharded, n_total, first_index, seed, dist)

    def _sharded(self, fn, n_total, first_index, seed, dist):
        bitmap = np.zeros((n_total + 7) // 8, np.uint8); digs = np.zeros(len(self.devices), np.uint64)
        total = C.c_uint64(); acc = C.c_uint64(); ms = C.c_float()
        rc = fn(self.h, C.c_uint64(n_total), C.c_uint64(first_index), C.c_uint64(seed), int(dist), C.c_void_p(bitmap.ctypes.data),
                C.c_void_p(digs.ctypes.data), C.byref(total), C.byref(acc), C.byref(ms))
        self._check(rc, fn.__name__)
        return dict(bitmap=bitmap, digests=digs, total_digest=int(total.value), accepted=int(acc.value), ms=float(ms.value))

    # ---- Fiat-Shamir, host arrays: the same bytes as the Context calls ----
    def prove_fs_batch(self, wit, rand, want_chal=True):
        """wit (12,n), rand (9,n) -> proof (27,n), status (n,) [, chal (6,n) = alpha beta gamma z v u]."""
        W = _Planes(wit, 12, name="wit"); n = W.n
        R = _Planes(rand, 9, n, "rand")
        proof = np.empty((27, n), np.uint8); status = np.empty((n,), np.uint8); chal = np.empty((6, n), np.uint8) if want_chal else None
        P = _Planes(proof, 27, n, "proof", out=True); S = _Planes(status, 1, n, "status", out=True)
        Ch = _Planes(chal, 6, n, "chal", out=True) if want_chal else None
        rc = self.lib.pbh_multi_prove_fs_batch(self.h, C.c_size_t(n), C.c_void_p(W.ptr), C.c_size_t(W.pitch), C.c_void_p(R.ptr),
                                               C.c_size_t(R.pitch), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(S.ptr),
                                               C.c_void_p(Ch.ptr if Ch else None), C.c_size_t(Ch.pitch if Ch else 0))
        self._check(rc, "pbh_multi_prove_fs_batch")
        return (proof, status, chal) if want_chal else (proof, status)

    def verify_fs_batch(self, proof, want_chal=False, want_gt=False):
        """proof (27,n) -> result (n,) [, chal (6,n)] [, gt (4,n)]."""
        P = _Planes(proof, 27, name="proof"); n = P.n
        result = np.empty((n,), np.uint8)
        chal = np.empty((6, n), np.uint8) if want_chal else None; gt = np.empty((4, n), np.uint8) if want_gt else None
        Rs = _Planes(result, 1, n, "result", out=True)
        Ch = _Planes(chal, 6, n, "chal", out=True) if want_chal else None; G = _Planes(gt, 4, n, "gt", out=True) if want_gt else None
        rc = self.lib.pbh_multi_verify_fs_batch(self.h, C.c_size_t(n), C.c_void_p(P.ptr), C.c_size_t(P.pitch), C.c_void_p(Rs.ptr),
                                                C.c_void_p(Ch.ptr if Ch else None), C.c_size_t(Ch.pitch if Ch else 0),
                                                C.c_void_p(G.ptr if G else None), C.c_size_t(G.pitch if G else 0))
        self._check(rc, "pbh_multi_verify_fs_batch")
        out = [result] + ([chal] if want_chal else []) + ([gt] if want_gt else [])
        return out[0] if len(out) == 1 else tuple(out)

    def prove_fs_packed(self, packed_in, want_chal_u=True):
        """PACKED_FS_WITNESS records -> PACKED_PROOF records [, challenge words]."""
        pin = Context._packed(packed_in, PACKED_FS_WITNESS, "packed_in"); n = pin.shape[0]
        out = np.zeros(n, dtype=PACKED_PROOF); cu = np.zeros(n, dtype="<u4") if want_chal_u else None
        self._check(self.lib.pbh_multi_prove_fs_packed(self.h, C.c_size_t(n), C.c_void_p(pin.ctypes.data), C.c_void_p(out.ctypes.data),
                                                       C.c_void_p(cu.ctypes.data if want_chal_u else None)), "pbh_multi_prove_fs_packed")
        return (out, cu) if want_chal_u else out

    def verify_fs_packed(self, proofs):
        prf = Context._packed(proofs, PACKED_PROOF, "proofs")
        res = np.zeros(prf.shape[0], dtype=np.uint8)
        self._check(self.lib.pbh_multi_verify_fs_packed(self.h, C.c_size_t(prf.shape[0]), C.c_void_p(prf.ctypes.data), C.c_void_p(res.ctypes.data)),
                    "pbh_multi_verify_fs_packed")
        return res


# ================================================================================================
# The reference's vocabulary (batch-of-1 wrappers)
# ================================================================================================
def f17(x):
    """src/pbh/mod.rs:13-16"""
    return int(x) % 17


def f101(x):
    """src/pbh/mod.rs:8-11"""
    return int(x) % 101


def g1f(x, y):
    """src/pbh/g1.rs:11-13 — an affine point; the identity is `None`."""
    return (f101(x), f101(y))


class Gate:
    """src/constraints.rs:10-64"""

    def __init__(self, q_l, q_r, q_o, q_m, q_c):
        self.q_l, self.q_r, self.q_o, self.q_m, self.q_c = f17(q_l), f17(q_r), f17(q_o), f17(q_m), f17(q_c)

    @classmethod
    def sum_a_b(cls): return cls(1, 1, -1, 0, 0)
    @classmethod
    def sub_a_b(cls): return cls(1, 1, 1, 0, 0)      # sic: identical signs in the reference (src/constraints.rs:37-45)
    @classmethod
    def mul_a_b(cls): return cls(0, 0, -1, 1, 0)
    @classmethod
    def bind_a(cls, value): return cls(1, 0, 0, 1, value)


class CopyOf:
    """src/constraints.rs:67-71"""

    def __init__(self, wire, n):
        self.wire, self.n = wire, n

    @classmethod
    def A(cls, n): return cls(0, n)
    @classmethod
    def B(cls, n): return cls(1, n)
    @classmethod
    def C(cls, n): return cls(2, n)


class Expression:
    """src/constraints.rs:246-287 — the reference's (unfinished) circuit front-end: an expression tree over named
    variables with `+`, `-`, `*`; `Constrains.eval_exprs` lowers it to gates.  Host-side only, as in the reference."""

    def __init__(self, kind, a=None, b=None):
        self.kind, self.a, self.b = kind, a, b

    @classmethod
    def Var(cls, name): return cls("var", name)
    @classmethod
    def Const(cls, value): return cls("const", f17(value))

    def __add__(self, rhs): return Expression("sum", self, rhs)      # src/constraints.rs:268-273
    def __sub__(self, rhs): return Expression("sub", self, rhs)      # :275-280
    def __mul__(self, rhs): return Expression("mul", self, rhs)      # :282-287

    def __str__(self):                                               # Display, src/constraints.rs:254-266
        if self.kind in ("var", "const"):
            return str(self.a)
        return "(%s%s%s)" % (self.a, {"sum": "+", "sub": "-", "mul": "*"}[self.kind], self.b)


class Constrains:
    """src/constraints.rs:109-153"""

    @staticmethod
    def eval_exprs(expr, variables, gates):
        """src/constraints.rs:155-196: post-order lowering.  `variables` maps a name to its index (a dict, in insertion
        order), `gates` collects (Gate, left index, right index, output index).  Returns the index holding the value of
        `expr`.  As in the reference a constant is not supported (`unimplemented!()`, :166-168), every operator node
        allocates a fresh variable "v<n>", and n is the number of variables at that moment."""
        if expr.kind == "var":
            return variables.setdefault(expr.a, len(variables))
        if expr.kind == "const":
            raise ReferencePanic(-1, "not implemented (src/constraints.rs:167)")
        l = Constrains.eval_exprs(expr.a, variables, gates)
        r = Constrains.eval_exprs(expr.b, variables, gates)
        n = len(variables)
        variables["v%d" % n] = n
        gates.append(({"mul": Gate.mul_a_b, "sum": Gate.sum_a_b, "sub": Gate.sub_a_b}[expr.kind](), l, r, n))
        return n

    def __init__(self, gates, copy_constraints):
        if len(gates) != 4:
            raise PbhError("this build mirrors the reference's prove(), which is hard-wired to 4 gates (src/plonk.rs:376-378)")
        self.gates = list(gates)
        self.c_a, self.c_b, self.c_c = copy_constraints

    def to_circuit(self):
        c = Circuit()
        for i, g in enumerate(self.gates):
            c.q_l[i], c.q_r[i], c.q_o[i], c.q_m[i], c.q_c[i] = g.q_l, g.q_r, g.q_o, g.q_m, g.q_c
        for name, vec in (("c_a", self.c_a), ("c_b", self.c_b), ("c_c", self.c_c)):
            for i, cp in enumerate(vec):
                getattr(c, name + "_wire")[i] = cp.wire
                getattr(c, name + "_index")[i] = cp.n
        return c


class Assigment:
    """src/constraints.rs:120-130"""

    def __init__(self, a, b, c):
        self.a, self.b, self.c = f17(a), f17(b), f17(c)


class Assigments:
    """src/constraints.rs:132-136, 233-244"""

    def __init__(self, assigments):
        self.a = [v.a for v in assigments]; self.b = [v.b for v in assigments]; self.c = [v.c for v in assigments]

    def __len__(self):
        return len(self.a)


class Challange:
    """src/plonk.rs:97-108"""

    def __init__(self, alpha, beta, gamma, z, v):
        self.alpha, self.beta, self.gamma, self.z, self.v = f17(alpha), f17(beta), f17(gamma), f17(z), f17(v)

    def column(self):
        return np.array([[self.alpha], [self.beta], [self.gamma], [self.z], [self.v]], dtype=np.uint8)


POINT_NAMES = "a_s b_s c_s z_s t_lo_s t_mid_s t_hi_s w_z_s w_z_omega_s".split()
EVAL_NAMES = "a_z b_z c_z s_sigma_1_z s_sigma_2_z r_z z_omega_z".split()


class Proof:
    """src/plonk.rs:61-95.  Points are (x, y) tuples, `None` for the identity."""

    def __init__(self, **kw):
        for name in POINT_NAMES + EVAL_NAMES:
            setattr(self, name, kw[name])

    def __eq__(self, other):
        return all(getattr(self, k) == getattr(other, k) for k in POINT_NAMES + EVAL_NAMES)

    def __repr__(self):
        return "Proof(" + ", ".join(f"{k}={getattr(self, k)}" for k in POINT_NAMES + EVAL_NAMES) + ")"

    def column(self):
        col = np.zeros((27, 1), dtype=np.uint8)
        for k, name in enumerate(POINT_NAMES):
            p = getattr(self, name)
            if p is None:
                p = (0, 0, 1)
            col[2 * k, 0], col[2 * k + 1, 0] = p[0], p[1]
            if len(p) > 2 and p[2]:
                if k < 8:
                    col[18, 0] |= 1 << k
                else:
                    col[19, 0] |= 1
        for k, name in enumerate(EVAL_NAMES):
            col[20 + k, 0] = getattr(self, name)
        return col

    @classmethod
    def from_column(cls, col):
        d = {}
        for k, name in enumerate(POINT_NAMES):
            inf = (col[18] >> k) & 1 if k < 8 else col[19] & 1
            x, y = int(col[2 * k]), int(col[2 * k + 1])
            d[name] = (None if (x == 0 and y == 0) else (x, y, 1)) if inf else (x, y)
        for k, name in enumerate(EVAL_NAMES):
            d[name] = int(col[20 + k])
        return cls(**d)


class SRS:
    """src/plonk.rs:28-48.  `SRS.create(s, n)` records the parameters; the points are computed by the context."""

    def __init__(self, s, n):
        self.s, self.n = f101(s), int(n)

    @classmethod
    def create(cls, s, n):
        return cls(s, n)


class Plonk:
    """src/plonk.rs:110-175, 191-650 — `Plonk.new(srs, omega_pows)`, then prove / verify one item on the GPU."""

    def __init__(self, srs, omega_pows, device=0, algo="table"):
        self.srs, self.omega_pows, self.device, self.algo = srs, f17(omega_pows), device, algo
        self._ctx = {}

    @classmethod
    def new(cls, srs, omega_pows, device=0, algo="table"):
        return cls(srs, omega_pows, device, algo)

    def _context(self, constraints):
        key = bytes(constraints.to_circuit())
        if key not in self._ctx:
            self._ctx[key] = Context(constraints.to_circuit(), self.srs.s, self.srs.n, self.omega_pows, self.device, self.algo)
        return self._ctx[key]

    def prove(self, constraints, assigments, challange, rand):
        ctx = self._context(constraints)
        wit = np.array([assigments.a + assigments.b + assigments.c], dtype=np.uint8).T.copy()
        rnd = np.array([[f17(r) for r in rand]], dtype=np.uint8).T.copy()
        proof, status = ctx.prove_batch(wit, rnd, challange.column())
        st = int(status[0])
        if st != ST_OK:
            raise ReferencePanic(st, PANIC_MESSAGES.get(st, f"status {st}"))
        return Proof.from_column(proof[:, 0])

    def verify(self, constraints, proof, challange, rand):
        ctx = self._context(constraints)
        res = ctx.verify_batch(proof.column(), challange.column(), np.array([f17(rand[0])], dtype=np.uint8))
        r = int(res[0])
        if r == VR_PANIC_ZH0:
            raise ReferencePanic(r, "called `Option::unwrap()` on a `None` value (src/plonk.rs:579)")
        if r == VR_BAD_ENCODING:
            raise ReferencePanic(r, "input byte outside the field (not representable in the reference)")
        return bool(r & 1)
