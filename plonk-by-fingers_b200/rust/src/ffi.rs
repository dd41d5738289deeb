//! Raw bindings to include/pbh_b200.h (libpbh_b200.so).  SOURCE ONLY: never compiled in this repository.
//! One declaration per C entry point the Rust surface (`crate::plonk`) or a batch caller needs; the header documents each.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_float, c_int, c_void};

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct pbh_circuit {
    pub q_l: [u8; 4], pub q_r: [u8; 4], pub q_o: [u8; 4], pub q_m: [u8; 4], pub q_c: [u8; 4],
    pub c_a_wire: [u8; 4], pub c_a_index: [u8; 4],
    pub c_b_wire: [u8; 4], pub c_b_index: [u8; 4],
    pub c_c_wire: [u8; 4], pub c_c_index: [u8; 4],
}
#[repr(C)]
pub struct pbh_ctx { _private: [u8; 0] }
#[repr(C)]
pub struct pbh_multi { _private: [u8; 0] }

// return codes
pub const PBH_OK: c_int = 0;
pub const PBH_ERR_BAD_ARGUMENT: c_int = -1;
pub const PBH_ERR_SETUP_PANIC: c_int = -2;
pub const PBH_ERR_CUDA: c_int = -3;
pub const PBH_ERR_NO_DEVICE: c_int = -4;
pub const PBH_ERR_UNSUPPORTED: c_int = -5;
// per-item prover status: the reference's panic sites in program order
pub const PBH_ST_OK: u8 = 0;
pub const PBH_ST_UNSATISFIED: u8 = 1;
pub const PBH_ST_ACC_DIV0: u8 = 2;
pub const PBH_ST_T_REMAINDER: u8 = 3;
pub const PBH_ST_T_SLICE: u8 = 4;
pub const PBH_ST_SRS_OOB: u8 = 5;
pub const PBH_ST_BAD_ENCODING: u8 = 32;
pub const PBH_ST_UNREPRESENTABLE: u8 = 33;
// per-item verifier result
pub const PBH_VR_ACCEPT: u8 = 0x01;
pub const PBH_VR_REJECT_PAIRING: u8 = 0x00;
pub const PBH_VR_NOT_ON_CURVE: u8 = 0x02;
pub const PBH_VR_NOT_IN_FIELD: u8 = 0x04;
pub const PBH_VR_PANIC_ZH0: u8 = 0x10;
pub const PBH_VR_BAD_ENCODING: u8 = 0x20;
pub const PBH_ALGO_ARITH: c_int = 0;
pub const PBH_ALGO_TABLE: c_int = 1;
pub const PBH_LANES: c_int = 4;

#[link(name = "pbh_b200")]
extern "C" {
    pub fn pbh_circuit_pbh_test(out: *mut pbh_circuit);
    pub fn pbh_ctx_create(circuit: *const pbh_circuit, srs_secret: u8, srs_n: u32, omega_pows: u8, device: c_int,
                          out: *mut *mut pbh_ctx) -> c_int;
    pub fn pbh_ctx_destroy(ctx: *mut pbh_ctx);
    pub fn pbh_last_error(ctx: *const pbh_ctx) -> *const c_char;
    pub fn pbh_ctx_set_algo(ctx: *mut pbh_ctx, algo: c_int) -> c_int;
    pub fn pbh_ctx_set_option(ctx: *mut pbh_ctx, option: c_int, value: c_int) -> c_int;
    pub fn pbh_ctx_sync(ctx: *mut pbh_ctx) -> c_int;
    pub fn pbh_ctx_stream(ctx: *mut pbh_ctx) -> *mut c_void;
    pub fn pbh_ctx_get_srs(ctx: *const pbh_ctx, g1s_xy_inf: *mut u8, cap_points: usize, n_points: *mut u32, g2: *mut u8) -> c_int;
    pub fn pbh_ctx_get_verifier_constants(ctx: *const pbh_ctx, selector_commits: *mut u8) -> c_int;
    // Plonk::prove / Plonk::verify over batches of byte planes, host pointers
    pub fn pbh_prove_batch(ctx: *mut pbh_ctx, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                           chal: *const u8, chal_pitch: usize, proof: *mut u8, proof_pitch: usize, status: *mut u8) -> c_int;
    pub fn pbh_verify_batch(ctx: *mut pbh_ctx, n: usize, proof: *const u8, proof_pitch: usize, chal: *const u8, chal_pitch: usize,
                            u: *const u8, result: *mut u8, gt: *mut u8, gt_pitch: usize) -> c_int;
    pub fn pbh_prove_verify_batch(ctx: *mut pbh_ctx, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                                  chal: *const u8, chal_pitch: usize, u: *const u8, proof: *mut u8, proof_pitch: usize,
                                  status: *mut u8, result: *mut u8) -> c_int;
    // asynchronous lanes over page-locked memory (two batches in flight keep both directions of the PCIe link busy)
    pub fn pbh_host_alloc(ctx: *mut pbh_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn pbh_host_alloc_input(ctx: *mut pbh_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn pbh_host_free(ctx: *mut pbh_ctx, ptr: *mut c_void) -> c_int;
    pub fn pbh_prove_batch_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8,
                                 rand_pitch: usize, chal: *const u8, chal_pitch: usize, proof: *mut u8, proof_pitch: usize,
                                 status: *mut u8) -> c_int;
    pub fn pbh_verify_batch_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, proof: *const u8, proof_pitch: usize, chal: *const u8,
                                  chal_pitch: usize, u: *const u8, result: *mut u8, gt: *mut u8, gt_pitch: usize) -> c_int;
    pub fn pbh_lane_sync(ctx: *mut pbh_ctx, lane: c_int) -> c_int;
    // Fiat-Shamir: challenges and the verifier's rand[0] derived on the device (include/pbh_b200.h)
    pub fn pbh_ctx_get_fs_seed(ctx: *const pbh_ctx, state_0: *mut u8) -> c_int;
    pub fn pbh_prove_fs_batch(ctx: *mut pbh_ctx, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                              proof: *mut u8, proof_pitch: usize, status: *mut u8, chal_out: *mut u8, chal_pitch: usize) -> c_int;
    pub fn pbh_verify_fs_batch(ctx: *mut pbh_ctx, n: usize, proof: *const u8, proof_pitch: usize, result: *mut u8,
                               chal_out: *mut u8, chal_pitch: usize, gt: *mut u8, gt_pitch: usize) -> c_int;
    // 32-byte records (Vec<Proof>-shaped exchange without per-field copies)
    pub fn pbh_prove_records(ctx: *mut pbh_ctx, n: usize, input: *const WitnessRecord, out: *mut ProofRecord) -> c_int;
    pub fn pbh_verify_records(ctx: *mut pbh_ctx, n: usize, proofs: *const ProofRecord, params: *const WitnessRecord,
                              result: *mut u8) -> c_int;
    // packed wire format: 16-byte prover inputs, 12-byte proofs, 4-byte challenge words (32 B up / 13 B down per proof + verification)
    pub fn pbh_prove_packed(ctx: *mut pbh_ctx, n: usize, input: *const PackedWitness, out: *mut PackedProof) -> c_int;
    pub fn pbh_verify_packed(ctx: *mut pbh_ctx, n: usize, proofs: *const PackedProof, chal_u: *const u32, result: *mut u8) -> c_int;
    pub fn pbh_prove_packed_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, input: *const PackedWitness, out: *mut PackedProof) -> c_int;
    pub fn pbh_verify_packed_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, proofs: *const PackedProof, chal_u: *const u32,
                                   result: *mut u8) -> c_int;
    pub fn pbh_prove_verify_packed(ctx: *mut pbh_ctx, n: usize, input: *const PackedWitness, out: *mut PackedProof, result: *mut u8) -> c_int;
    pub fn pbh_prove_verify_packed_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, input: *const PackedWitness, out: *mut PackedProof,
                                         result: *mut u8) -> c_int;
    // host-side format conversion (CPU loops, no device): build packed records from byte planes and read proofs back
    pub fn pbh_pack_witness_host(n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize, chal: *const u8,
                                 chal_pitch: usize, u: *const u8, out: *mut PackedWitness) -> c_int;
    pub fn pbh_unpack_witness_host(n: usize, input: *const PackedWitness, wit: *mut u8, wit_pitch: usize, rand: *mut u8, rand_pitch: usize,
                                   chal: *mut u8, chal_pitch: usize, u: *mut u8) -> c_int;
    pub fn pbh_pack_chal_u_host(n: usize, chal: *const u8, chal_pitch: usize, u: *const u8, out: *mut u32) -> c_int;
    pub fn pbh_pack_proofs_host(n: usize, proof: *const u8, proof_pitch: usize, status: *const u8, out: *mut PackedProof) -> c_int;
    pub fn pbh_unpack_proofs_host(n: usize, input: *const PackedProof, proof: *mut u8, proof_pitch: usize, status: *mut u8) -> c_int;
    // Fiat-Shamir over packed records: 12-byte prover inputs (wit + rand), 12-byte proofs, optional 4-byte derived challenge words
    pub fn pbh_prove_fs_packed(ctx: *mut pbh_ctx, n: usize, input: *const PackedFsWitness, out: *mut PackedProof, chal_u_out: *mut u32) -> c_int;
    pub fn pbh_verify_fs_packed(ctx: *mut pbh_ctx, n: usize, proofs: *const PackedProof, result: *mut u8) -> c_int;
    pub fn pbh_prove_fs_packed_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, input: *const PackedFsWitness, out: *mut PackedProof,
                                     chal_u_out: *mut u32) -> c_int;
    pub fn pbh_verify_fs_packed_async(ctx: *mut pbh_ctx, lane: c_int, n: usize, proofs: *const PackedProof, result: *mut u8) -> c_int;
    pub fn pbh_prove_fs_packed_dev(ctx: *mut pbh_ctx, n: usize, input: *const PackedFsWitness, out: *mut PackedProof,
                                   chal_u_out: *mut u32) -> c_int;
    pub fn pbh_verify_fs_packed_dev(ctx: *mut pbh_ctx, n: usize, proofs: *const PackedProof, result: *mut u8) -> c_int;
    pub fn pbh_pack_fs_witness_host(n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                                    out: *mut PackedFsWitness) -> c_int;
    pub fn pbh_unpack_fs_witness_host(n: usize, input: *const PackedFsWitness, wit: *mut u8, wit_pitch: usize, rand: *mut u8,
                                      rand_pitch: usize) -> c_int;
    // batched equivalents of the crate's value-type operations (a selection; the header has them all)
    pub fn pbh_kzg_commit_batch(ctx: *mut pbh_ctx, n: usize, coeffs: *const u8, in_pitch: usize, out: *mut u8, out_pitch: usize,
                                on_device: c_int) -> c_int;                       // SRS::eval_at_s
    pub fn pbh_pairing_batch(ctx: *mut pbh_ctx, n: usize, input: *const u8, in_pitch: usize, out: *mut u8, out_pitch: usize,
                             on_device: c_int) -> c_int;                          // PBHPairing::pairing
    pub fn pbh_mul_ntt_batch(ctx: *mut pbh_ctx, n: usize, modulus: u32, omega: u32, la: u32, lb: u32, a: *const u16, a_pitch: usize,
                             b: *const u16, b_pitch: usize, out: *mut u16, out_pitch: usize, on_device: c_int) -> c_int;  // fft::mul_ntt
    pub fn pbh_coset_ntt4_batch(ctx: *mut pbh_ctx, n: usize, k: u32, coeffs: *const u8, in_pitch: usize, evals: *mut u8,
                                out_pitch: usize, on_device: c_int) -> c_int;     // evaluations on k1_h / k2_h (src/plonk.rs:136-139)
    pub fn pbh_coset_intt4_batch(ctx: *mut pbh_ctx, n: usize, k: u32, evals: *const u8, in_pitch: usize, coeffs: *mut u8,
                                 out_pitch: usize, on_device: c_int) -> c_int;
    // several GPUs from one process: contiguous shards, one in-library ncclAllGather of verdict bitmaps + digests
    pub fn pbh_multi_create(circuit: *const pbh_circuit, srs_secret: u8, srs_n: u32, omega_pows: u8, devices: *const c_int,
                            n_dev: c_int, out: *mut *mut pbh_multi) -> c_int;
    pub fn pbh_multi_destroy(m: *mut pbh_multi);
    pub fn pbh_multi_device_count(m: *const pbh_multi) -> c_int;
    pub fn pbh_multi_ctx(m: *mut pbh_multi, i: c_int) -> *mut pbh_ctx;
    pub fn pbh_multi_last_error(m: *const pbh_multi) -> *const c_char;
    pub fn pbh_multi_set_algo(m: *mut pbh_multi, algo: c_int) -> c_int;
    pub fn pbh_multi_prove_batch(m: *mut pbh_multi, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                                 chal: *const u8, chal_pitch: usize, proof: *mut u8, proof_pitch: usize, status: *mut u8) -> c_int;
    pub fn pbh_multi_verify_batch(m: *mut pbh_multi, n: usize, proof: *const u8, proof_pitch: usize, chal: *const u8,
                                  chal_pitch: usize, u: *const u8, result: *mut u8, gt: *mut u8, gt_pitch: usize) -> c_int;
    pub fn pbh_multi_prove_packed(m: *mut pbh_multi, n: usize, input: *const PackedWitness, out: *mut PackedProof) -> c_int;
    pub fn pbh_multi_verify_packed(m: *mut pbh_multi, n: usize, proofs: *const PackedProof, chal_u: *const u32, result: *mut u8) -> c_int;
    // peer windows: the shard summaries stored into every peer's buffer by the kernels that produce them
    pub fn pbh_window_create(ctx: *mut pbh_ctx, bytes_per_rank: usize, rank: c_int, world: c_int, base_out: *mut *mut c_void,
                             handle_out: *mut u8) -> c_int;
    pub fn pbh_window_attach(ctx: *mut pbh_ctx, handles: *const u8) -> c_int;
    pub fn pbh_window_attach_ptrs(ctx: *mut pbh_ctx, bases: *const *mut c_void) -> c_int;
    pub fn pbh_window_share(owner: *mut pbh_ctx, other: *mut pbh_ctx) -> c_int;
    pub fn pbh_window_destroy(ctx: *mut pbh_ctx) -> c_int;
    pub fn pbh_multi_prove_verify_sharded(m: *mut pbh_multi, n_total: u64, first_index: u64, seed: u64, dist: c_int,
                                          bitmap_out: *mut u8, digests_out: *mut u64, total_digest_out: *mut u64,
                                          accepted_out: *mut u64, ms_out: *mut c_float) -> c_int;
    // Fiat-Shamir shard summaries (device pointers, compute stream) and the Fiat-Shamir multi-device calls
    pub fn pbh_prove_fs_digest_batch_dev(ctx: *mut pbh_ctx, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                                         proof: *mut u8, proof_pitch: usize, status: *mut u8, chal_out: *mut u8, chal_pitch: usize,
                                         first_index: u64, digest: *mut u64) -> c_int;
    pub fn pbh_verify_fs_bitmap_batch_dev(ctx: *mut pbh_ctx, n: usize, proof: *const u8, proof_pitch: usize, result: *mut u8,
                                          bitmap: *mut u8) -> c_int;
    pub fn pbh_multi_prove_fs_batch(m: *mut pbh_multi, n: usize, wit: *const u8, wit_pitch: usize, rand: *const u8, rand_pitch: usize,
                                    proof: *mut u8, proof_pitch: usize, status: *mut u8, chal_out: *mut u8, chal_pitch: usize) -> c_int;
    pub fn pbh_multi_verify_fs_batch(m: *mut pbh_multi, n: usize, proof: *const u8, proof_pitch: usize, result: *mut u8,
                                     chal_out: *mut u8, chal_pitch: usize, gt: *mut u8, gt_pitch: usize) -> c_int;
    pub fn pbh_multi_prove_fs_packed(m: *mut pbh_multi, n: usize, input: *const PackedFsWitness, out: *mut PackedProof,
                                     chal_u_out: *mut u32) -> c_int;
    pub fn pbh_multi_verify_fs_packed(m: *mut pbh_multi, n: usize, proofs: *const PackedProof, result: *mut u8) -> c_int;
    pub fn pbh_multi_prove_verify_fs_sharded(m: *mut pbh_multi, n_total: u64, first_index: u64, seed: u64, dist: c_int,
                                             bitmap_out: *mut u8, digests_out: *mut u64, total_digest_out: *mut u64,
                                             accepted_out: *mut u64, ms_out: *mut c_float) -> c_int;
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct WitnessRecord { pub wit: [u8; 12], pub rand: [u8; 9], pub chal: [u8; 5], pub u: u8, pub reserved: [u8; 5] }
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct ProofRecord { pub xy: [u8; 18], pub inf_lo: u8, pub inf_hi: u8, pub evals: [u8; 7], pub status: u8, pub reserved: [u8; 4] }
#[repr(C)]
#[derive(Clone, Copy, Default, PartialEq, Eq, Debug)]
pub struct PackedWitness { pub w: [u32; 4] }
#[repr(C)]
#[derive(Clone, Copy, Default, PartialEq, Eq, Debug)]
pub struct PackedProof { pub points_lo: u32, pub points_hi: u32, pub evals_status: u32 }
#[repr(C)]
#[derive(Clone, Copy, Default, PartialEq, Eq, Debug)]
pub struct PackedFsWitness { pub w: [u32; 3] }
