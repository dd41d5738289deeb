/* pbh_b200.h — C ABI of the B200-native batched Plonk-by-hand prover / verifier.
 *
 * This is the drop-in boundary for the hot path of adria0/plonk-by-fingers.  The reference has no
 * FFI of its own: its boundary is the crate's public Rust API (SURVEY.md §8b).  Each entry point
 * below names the reference function(s) whose results it reproduces bit for bit (file:line relative
 * to the reference repository).  The Rust-side binding a maintainer would add is in INTEGRATION.md
 * and plonk-by-fingers_b200/rust/.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Return 0 on success, a negative pbh_error otherwise; nothing
 *    aborts or unwinds across this boundary.  A Rust panic of the reference becomes a per-item
 *    status byte (below), never a process abort.
 *  - One context drives one CUDA device (one process per GPU under torchrun; pbh_multi_* below drives several devices
 *    from one process).  A context may be used from one host thread at a time.  Launches recorded into CUDA graphs
 *    (stream capture around `_dev` calls) each hold a tile-scheduler slot for the life of the context (32768 per
 *    context), and a graph must not be replayed concurrently with itself.
 *  - Batches are structure-of-arrays BYTE PLANES: plane k of an n-item batch is the n bytes at
 *    base + k*pitch (pitch >= n; pitch is in bytes and lets a shard address a column range of a
 *    larger batch without repacking).  One byte per field element: F_17 values 0..16, F_101
 *    values 0..100.
 *  - Entry points without suffix take HOST pointers and run H2D -> kernels -> D2H on the context's
 *    streams (chunked and overlapped).  `_dev` variants take DEVICE pointers on the context's
 *    device and only enqueue kernels on the context's compute stream (use pbh_ctx_sync to wait).
 *
 * Encoding of out-of-range bytes.  The reference cannot represent them (`U64Field` values are
 * only constructible through `From<u64>`/`f17`/`f101`, which reduce): a witness, blinder, challenge
 * or `u` byte >= 17, or a G1 coordinate byte >= 101, or an infinity-bitmap bit outside the 9 defined
 * ones, yields status PBH_ST_BAD_ENCODING for that item.  The seven proof evaluations are the one
 * exception: a byte >= 17 there models a failing `in_field()` (src/plonk.rs:538-547) and yields a
 * completed verification with verdict false / PBH_VR_NOT_IN_FIELD, after the on-curve check as in
 * the reference.
 */
#ifndef PBH_B200_H
#define PBH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: round 2 added entry points only (lanes, packed records, peer windows, multi-device, sweeps); every round-1 signature is unchanged
 * 3: entry points added (Fiat-Shamir over packed records), none changed
 * 4: entry points added (Fiat-Shamir shard summaries and multi-device calls), none changed */
#define PBH_ABI_VERSION 4

/* ---- errors (return values) ---------------------------------------------------------------- */
typedef enum pbh_error {
  PBH_OK = 0,
  PBH_ERR_BAD_ARGUMENT = -1,   /* null pointer, pitch < n, unsupported size, ... */
  PBH_ERR_SETUP_PANIC = -2,    /* the reference's SRS::create / Plonk::new would panic on these inputs */
  PBH_ERR_CUDA = -3,           /* a CUDA call failed; see pbh_last_error */
  PBH_ERR_NO_DEVICE = -4,      /* no usable CUDA device: there is NO CPU fallback */
  PBH_ERR_UNSUPPORTED = -5
} pbh_error;

/* ---- per-item prover status (mirrors the reference's panic sites in program order) ----------- */
#define PBH_ST_OK 0            /* proof bytes are valid                                            */
#define PBH_ST_UNSATISFIED 1   /* src/plonk.rs:199  assert!(constraints.satisfies(assigments))      */
#define PBH_ST_ACC_DIV0 2      /* src/plonk.rs:297  (dend / dsor).unwrap()                          */
#define PBH_ST_T_REMAINDER 3   /* src/plonk.rs:370  assert_eq!(rem, Poly::zero())  (Q1)             */
#define PBH_ST_T_SLICE 4       /* src/plonk.rs:376  t_x.coeffs()[12..18]           (Q5)             */
#define PBH_ST_SRS_OOB 5       /* src/plonk.rs:56   g1s[n] out of bounds           (Q2)             */
#define PBH_ST_BAD_ENCODING 32 /* input byte outside the field (not representable in the reference) */
#define PBH_ST_UNREPRESENTABLE 33 /* only from the packed-format helpers: this proof has no packed form (see below) */

/* ---- per-item verifier result byte ------------------------------------------------------------ */
#define PBH_VR_ACCEPT 0x01        /* verify() == true                      src/plonk.rs:649         */
#define PBH_VR_REJECT_PAIRING 0x00 /* verify() == false: e_1 != e_2        src/plonk.rs:649         */
#define PBH_VR_NOT_ON_CURVE 0x02  /* verify() == false at Step 1           src/plonk.rs:523-534     */
#define PBH_VR_NOT_IN_FIELD 0x04  /* verify() == false at Step 2           src/plonk.rs:538-547     */
#define PBH_VR_PANIC_ZH0 0x10     /* verify() panics: Z_H(z) == 0          src/plonk.rs:579         */
#define PBH_VR_BAD_ENCODING 0x20  /* see "Encoding of out-of-range bytes"                           */
/* bit 0 of the result byte is the reference's bool whenever bits 4 and 5 are clear. */

/* ---- wire layout (plane indices) ------------------------------------------------------------ */
/* prover input: src/plonk.rs:191-197 — Assigments (12) + rand[9] + Challange (5) = 26 planes      */
#define PBH_WIT_PLANES 12   /* a[0..4), b[0..4), c[0..4)          src/constraints.rs:132-136        */
#define PBH_RAND_PLANES 9   /* b1..b9                             src/plonk.rs:196, 248, 267        */
#define PBH_CHAL_PLANES 5   /* alpha, beta, gamma, z, v           src/plonk.rs:97-108               */
/* proof: src/plonk.rs:61-95 — 9 G1 points then 7 F_17 evaluations                                 */
#define PBH_PROOF_POINTS 9  /* a_s b_s c_s z_s t_lo_s t_mid_s t_hi_s w_z_s w_z_omega_s              */
#define PBH_PROOF_EVALS 7   /* a_z b_z c_z s_sigma_1_z s_sigma_2_z r_z z_omega_z                    */
/* planes 0..17: x,y of point k at planes 2k, 2k+1; planes 18,19: `infinite` flags (bit k of plane
 * 18 for points 0..7, bit 0 of plane 19 for point 8); planes 20..26: the evaluations.            */
#define PBH_PROOF_PLANES 27
#define PBH_PROOF_INF_PLANE 18
#define PBH_PROOF_EVAL_PLANE 20
/* algorithmic bytes per item (SURVEY.md §8d): prove 26 in + 27 proof + 1 status = 54;
 * verify 27 + 5 + 1 in + 1 result = 34                                                            */
#define PBH_PROVE_BYTES_PER_ITEM 54
#define PBH_VERIFY_BYTES_PER_ITEM 34

/* ---- circuit description: src/constraints.rs:109-118 (Constrains) ---------------------------- */
#define PBH_N_GATES 4       /* prove() is hard-wired to 4 gates: src/plonk.rs:376-378              */
#define PBH_COPY_A 0
#define PBH_COPY_B 1
#define PBH_COPY_C 2
typedef struct pbh_circuit {
  /* selector vectors, F_17 values: src/constraints.rs:110-114 */
  uint8_t q_l[PBH_N_GATES], q_r[PBH_N_GATES], q_o[PBH_N_GATES], q_m[PBH_N_GATES], q_c[PBH_N_GATES];
  /* copy constraints CopyOf::{A,B,C}(n): wire = PBH_COPY_*, index = n (1-based): :67-71, :115-117 */
  uint8_t c_a_wire[PBH_N_GATES], c_a_index[PBH_N_GATES];
  uint8_t c_b_wire[PBH_N_GATES], c_b_index[PBH_N_GATES];
  uint8_t c_c_wire[PBH_N_GATES], c_c_index[PBH_N_GATES];
} pbh_circuit;

/* algorithm selection for the group operations of the fused kernels (both are bit-exact) */
#define PBH_ALGO_ARITH 0  /* per-item affine curve arithmetic, Miller loop and final exponentiation */
#define PBH_ALGO_TABLE 1  /* group-structure tables built at context creation by the ARITH kernels  */

typedef struct pbh_ctx pbh_ctx;

/* The circuit of the reference's only end-to-end test (src/pbh/mod.rs:56-67). */
void pbh_circuit_pbh_test(pbh_circuit* out);

/* SRS::create(s, srs_n) (src/plonk.rs:35-48) + Plonk::new(srs, omega_pows) (src/plonk.rs:120-175)
 * + the circuit-constant work the reference redoes on every call (src/plonk.rs:222-243, 328-333,
 * 506-517, 557-562), computed once and uploaded to `device`.  omega_pows must be 4.
 * PBH_ERR_SETUP_PANIC when the reference would panic (e.g. s = 0, or G2 * s hitting P + (-P)). */
int pbh_ctx_create(const pbh_circuit* circuit, uint8_t srs_secret, uint32_t srs_n, uint8_t omega_pows,
                   int device, pbh_ctx** out);
void pbh_ctx_destroy(pbh_ctx* ctx);
const char* pbh_last_error(const pbh_ctx* ctx);   /* ctx may be NULL: last global (creation) error */
int pbh_ctx_set_algo(pbh_ctx* ctx, int algo);     /* PBH_ALGO_* ; default PBH_ALGO_TABLE            */
int pbh_ctx_get_algo(const pbh_ctx* ctx);
/* Tuning switches (results never change).  PBH_OPT_PROVER_FP32: with PBH_ALGO_TABLE, run the prover's F_17
 * arithmetic as exact small-integer FP32 on the FMA pipes (1, default) or as int32 IMAD arithmetic (0).  The verifier
 * has its own switch, PBH_OPT_VERIFIER_FP32. */
#define PBH_OPT_PROVER_FP32 1
/* PBH_OPT_PROVER_LAUNCH_SHAPE: threads x min-resident-blocks of the FP32 prover: 0 = 256x2 (default), 1 = 256x1,
 * 2 = 128x4, 3 = 128x5, 4 = 128x6 (register budget 128 / 255 / 128 / 96 / 80 per thread) */
#define PBH_OPT_PROVER_LAUNCH_SHAPE 2
/* PBH_OPT_TMA: stage 256-item tiles through shared memory with TMA bulk tensor copies (1, default; used when every
 * base pointer and pitch is a multiple of 16 bytes) or use plain per-thread loads and stores (0). */
#define PBH_OPT_TMA 3
/* PBH_OPT_CHUNK_LOG2: log2 of the items per staged chunk of the host-pointer entry points (8..20, default 18: measured best on PCIe Gen5). */
#define PBH_OPT_CHUNK_LOG2 4
/* PBH_OPT_SPECIALISE: when the context is the reference's own test circuit with SRS::create(2, 6), run the prover
 * instantiation whose circuit and SRS constants are compile-time (1, default) or the generic kernel (0). */
#define PBH_OPT_SPECIALISE 5
/* PBH_OPT_HOST_DIRECT: when EVERY buffer of pbh_prove_batch / pbh_verify_batch is page-locked and mapped
 * (cudaHostAlloc, cudaHostRegister), run the kernel in place on the caller's memory - its tile loads and stores cross
 * PCIe directly - instead of staging chunks through device buffers (1, default; 0 = always stage).  Pageable buffers
 * always take the staged path. */
#define PBH_OPT_HOST_DIRECT 6
/* PBH_OPT_VERIFIER_FP32: with PBH_ALGO_TABLE, run the verifier's F_17 scalar work in int32 (0, default: measured 25.4
 * against 28.7 us per 2^20 items) or as exact small-integer FP32 (1). */
#define PBH_OPT_VERIFIER_FP32 7
/* PBH_OPT_LANE_MODE: how the asynchronous lane calls (pbh_prove_batch_async / pbh_verify_batch_async) move page-locked
 * buffers.  Bit 0: inputs are uploaded whole by the copy engine into a per-lane staging buffer (else the kernel reads mapped
 * memory in place); bit 1: outputs come back through the copy engine (else the kernel stores into mapped memory in place).
 * 0 = in place both ways, 1 = copy-engine upload + in-place stores, 3 = copy engine both ways (default: measured 1.28 ms per
 * 2^20 prove + verify pairs on PCIe Gen5 x16, i.e. the upload link at 48 GB/s, against 1.33 ms for mode 1 and 1.48 ms for 0).  Buffers that are page-locked but not mapped always go through the copy engine. */
#define PBH_OPT_LANE_MODE 8
/* PBH_OPT_HOST_STAGE: PAGEABLE caller memory (a plain Vec<u8> / malloc) in the synchronous host-pointer calls is staged by the
 * library itself - a small pool of host threads copies row segments between the caller's memory and page-locked mirrors of
 * the staging buffers, which the copy engines then move asynchronously - (1, default) or left to the driver's own staging
 * of pageable copies, which runs on the calling thread at about 12 GB/s (0).  Page-locked memory never takes this path. */
#define PBH_OPT_HOST_STAGE 9
/* PBH_OPT_PROOF_RESIDENT: when pbh_verify_packed_async is called on a lane for the very `out` buffer (same pointer, same n) that the
 * immediately preceding call on that lane, pbh_prove_packed_async, is still filling - no pbh_lane_sync / pbh_ctx_sync and no other
 * call on the lane in between, so by the lane contract the caller cannot have touched the buffer and its contents will be exactly
 * what the device holds - the verifier reads the device-resident copy of those proofs instead of uploading them again (1,
 * default); the proofs still travel to the host as the prove call's output.  0 = always upload what the host buffer holds.
 * Results are identical either way. */
#define PBH_OPT_PROOF_RESIDENT 10
int pbh_ctx_set_option(pbh_ctx* ctx, int option, int value);
int pbh_ctx_device(const pbh_ctx* ctx);
int pbh_ctx_sync(pbh_ctx* ctx);                   /* wait for everything enqueued on the context    */
/* CUDA stream handle (cudaStream_t) the `_dev` entry points launch on; for event timing. */
void* pbh_ctx_stream(pbh_ctx* ctx);
/* number of kernel launches issued through this context so far */
uint64_t pbh_ctx_launch_count(const pbh_ctx* ctx);

/* Read back setup results (host copies): the SRS of src/plonk.rs:28-32 and the hoisted constants.
 * g1s_xy_inf: srs_n+1 triples (x,y,infinite); g2: g2_1.a, g2_1.b, g2_s.a, g2_s.b;
 * selector_commits: q_m_s q_l_s q_r_s q_o_s q_c_s sigma_1_s sigma_2_s sigma_3_s as triples. */
int pbh_ctx_get_srs(const pbh_ctx* ctx, uint8_t* g1s_xy_inf, size_t g1s_capacity_points, uint32_t* n_points,
                    uint8_t g2[4]);
int pbh_ctx_get_verifier_constants(const pbh_ctx* ctx, uint8_t selector_commits[24]);

/* Plonk::prove (src/plonk.rs:191-466), n items.
 *   wit   12 planes, rand 9 planes, chal 5 planes (each with its own pitch)
 *   proof 27 planes (zeroed for items whose status != PBH_ST_OK), status n bytes */
int pbh_prove_batch(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand,
                    size_t rand_pitch, const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch,
                    uint8_t* status);
int pbh_prove_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand,
                        size_t rand_pitch, const uint8_t* chal, size_t chal_pitch, uint8_t* proof,
                        size_t proof_pitch, uint8_t* status);

/* Plonk::verify (src/plonk.rs:468-650), n items.
 *   proof 27 planes, chal 5 planes, u n bytes (rand[0] of :473)
 *   result n bytes of PBH_VR_*; gt (nullable) 4 planes e_1.a e_1.b e_2.a e_2.b, defined when the
 *   pairing check was reached (result is ACCEPT or REJECT_PAIRING), zero otherwise. */
int pbh_verify_batch(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                     size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch);
int pbh_verify_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                         size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch);

/* ---- asynchronous host-pointer calls: lanes ---------------------------------------------------------------------------
 * Same arguments and results as pbh_prove_batch / pbh_verify_batch, but the call only ENQUEUES the work on lane `lane`
 * (0 .. PBH_LANES-1) and returns.  Calls on one lane run in issue order, so verify(k) may read the proof that prove(k)
 * writes when both use the same lane; calls on different lanes overlap - PCIe is full duplex, the download of one batch
 * travels beside the upload of the next.  Every buffer must stay valid and untouched until pbh_lane_sync(ctx, lane) or
 * pbh_ctx_sync(ctx) returns.  Only page-locked buffers (pbh_host_alloc, cudaHostAlloc, cudaHostRegister) are asynchronous
 * (PBH_OPT_LANE_MODE says how they travel); with pageable memory the call waits for the context's earlier work and then
 * behaves exactly like the synchronous entry point.  Batches above 2^24 items are processed synchronously as well.
 * Every lane call (the _async entry points here and below) has one failure policy: a call that fails after it has enqueued
 * copies of the caller's buffers waits for its lane before it returns the error, so the buffers may be released or reused as
 * soon as a failed call has returned. */
#define PBH_LANES 4
int pbh_prove_batch_async(pbh_ctx* ctx, int lane, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand,
                          size_t rand_pitch, const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch,
                          uint8_t* status);
int pbh_verify_batch_async(pbh_ctx* ctx, int lane, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                           size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch);
int pbh_lane_sync(pbh_ctx* ctx, int lane);

/* Page-locked, mapped host memory for the host-pointer entry points (they then run in place on it, see
 * PBH_OPT_HOST_DIRECT).  When the platform exposes the NUMA node of the device's PCIe root (sysfs; pbh_ctx_numa_node
 * returns it, -1 otherwise) the pages are bound to that node before they are locked.  Freed by pbh_host_free or with the
 * context. */
int pbh_host_alloc(pbh_ctx* ctx, size_t bytes, void** out);
/* The same as write-combined memory, for INPUT buffers only (the host writes them sequentially, the device reads them): device
 * reads need no snoop of the CPU caches.  CPU reads of such memory are uncached and slow. */
int pbh_host_alloc_input(pbh_ctx* ctx, size_t bytes, void** out);
int pbh_host_free(pbh_ctx* ctx, void* ptr);
int pbh_ctx_numa_node(const pbh_ctx* ctx);

/* Extension (no counterpart in the reference): Plonk::prove followed by Plonk::verify of the fresh proofs with
 * challenge `chal` and rand[0] = u, host pointers.  Same bytes as pbh_prove_batch + pbh_verify_batch, but a proof
 * produced on the device does not cross PCIe twice.  Items whose status != PBH_ST_OK have a zeroed proof, for which
 * verify answers PBH_VR_NOT_ON_CURVE. */
int pbh_prove_verify_batch(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand,
                           size_t rand_pitch, const uint8_t* chal, size_t chal_pitch, const uint8_t* u, uint8_t* proof,
                           size_t proof_pitch, uint8_t* status, uint8_t* result);

/* ---- Fiat-Shamir transcript — SURVEY.md §8(f) row 1 -------------------------------------------------------------
 * The reference leaves the five challenges and the verifier's rand[0] to the caller (src/plonk.rs:195, 201-206, 472-473,
 * 519).  These entry points derive them on the device, so a batch needs no host-made challenges.  Everything else is
 * Plonk::prove / Plonk::verify unchanged: a Fiat-Shamir proof is exactly the proof pbh_prove_batch returns when it is
 * handed the derived challenges, with the same status byte, and pbh_verify_fs_batch answers what pbh_verify_batch
 * answers for the derived challenges and u.
 *
 * PARITY UNPINNED BY THE REFERENCE: the reference has no transcript, so no vector of its own pins these two entry points.  What
 * is pinned: both SHA-256 implementations against hashlib, the oracle's challenges against a replay of this specification from the
 * proof bytes alone, and - the part the reference does pin - that the proof / verdict equal Plonk::prove / Plonk::verify handed
 * the derived challenges (tests/test_fiat_shamir.py).
 *
 * Transcript.  A state is 32 bytes; state_{k+1} = SHA-256(state_k || message_k) (FIPS 180-4; every message is at most
 * 12 bytes, so each step is a single compression).  A G1 point is absorbed as the four bytes (x, y, infinite as 0/1, 0),
 * an evaluation as its byte.  A challenge is a big-endian 64-bit slice of the new state reduced mod 17.
 *   state_0 = SHA-256("plonk-by-fingers/fiat-shamir/v1" || omega_pows || the 44 bytes of pbh_circuit in declaration
 *             order || number of SRS points || the SRS points (4 bytes each) || g2_1.a g2_1.b g2_s.a g2_s.b)
 *   state_1 = H(state_0 || a_s b_s c_s)                 beta  = bytes 0..7 of state_1 mod 17, gamma = bytes 8..15 mod 17
 *   state_2 = H(state_1 || z_s)                         alpha = bytes 0..7 of state_2 mod 17
 *   state_3 = H(state_2 || t_lo_s t_mid_s t_hi_s)       z     = bytes 0..7 of state_3 mod 17
 *   state_4 = H(state_3 || a_z b_z c_z s_sigma_1_z s_sigma_2_z r_z z_omega_z)          v = bytes 0..7 of state_4 mod 17
 *   state_5 = H(state_4 || w_z_s w_z_omega_s)           u     = bytes 0..7 of state_5 mod 17
 * The prover asks for each challenge where the reference first uses it (beta, gamma: src/plonk.rs:283; alpha: :343;
 * z: :393; v: :430), so a proof that panics early never needs the later ones.  The reference's quirks are kept: most
 * uniformly drawn challenges end in one of its panics (SURVEY.md §2.4), reported in the status byte as usual.
 * chal_out (nullable): 6 planes alpha beta gamma z v u; zero for items whose status != PBH_ST_OK (prove) or whose
 * result is PBH_VR_BAD_ENCODING (verify). */
#define PBH_FS_CHAL_PLANES 6
int pbh_ctx_get_fs_seed(const pbh_ctx* ctx, uint8_t state_0[32]);
int pbh_prove_fs_batch(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand, size_t rand_pitch,
                       uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch);
int pbh_prove_fs_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand, size_t rand_pitch,
                           uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch);
/* proof 27 planes in; result n bytes of PBH_VR_*; gt (nullable) as in pbh_verify_batch */
int pbh_verify_fs_batch(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result, uint8_t* chal_out,
                        size_t chal_pitch, uint8_t* gt, size_t gt_pitch);
int pbh_verify_fs_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result, uint8_t* chal_out,
                            size_t chal_pitch, uint8_t* gt, size_t gt_pitch);
/* The same two calls over packed records: "Fiat-Shamir over packed records" below. */

/* ---- record (array-of-structs) wire format — SURVEY.md §8(f) row 3 ---------------------------------------------
 * The reference has no serialisation (Proof only derives Debug, PartialEq: src/plonk.rs:61).  These 32-byte records let a
 * host exchange `Vec<Proof>` / per-item inputs with the library without per-field copies; the library transposes between
 * records and byte planes on the device. */
typedef struct pbh_witness_record {  /* one prove / verify input: Assigments + rand + Challange (src/plonk.rs:191-197, 468-474) */
  uint8_t wit[12];      /* a[0..4) b[0..4) c[0..4) */
  uint8_t rand[9];      /* b1..b9 */
  uint8_t chal[5];      /* alpha beta gamma z v */
  uint8_t u;            /* verifier rand[0] */
  uint8_t reserved[5];  /* ignored on input */
} pbh_witness_record;
typedef struct pbh_proof_record {    /* one Proof (src/plonk.rs:61-95) + its status */
  uint8_t xy[18];       /* x, y of a_s b_s c_s z_s t_lo_s t_mid_s t_hi_s w_z_s w_z_omega_s */
  uint8_t inf_lo, inf_hi; /* `infinite` flags: bit k of inf_lo for points 0..7, bit 0 of inf_hi for point 8 */
  uint8_t evals[7];     /* a_z b_z c_z s_sigma_1_z s_sigma_2_z r_z z_omega_z */
  uint8_t status;       /* PBH_ST_* (written by prove, ignored by verify) */
  uint8_t reserved[4];  /* written as zero */
} pbh_proof_record;
/* Plonk::prove over n records (host pointers): out[i] = proof and status of in[i]. */
int pbh_prove_records(pbh_ctx* ctx, size_t n, const pbh_witness_record* in, pbh_proof_record* out);
/* Plonk::verify over n records (host pointers): proofs[i] checked with params[i].chal and params[i].u; result n bytes of PBH_VR_*. */
int pbh_verify_records(pbh_ctx* ctx, size_t n, const pbh_proof_record* proofs, const pbh_witness_record* params, uint8_t* result);
/* Device-side transposes between records and byte planes (device pointers).  Null plane pointers are skipped.
 * witness records <-> wit (12 planes), rand (9), chal (5), u (1); proof records <-> proof (27 planes), status (1). */
int pbh_witness_records_to_planes_dev(pbh_ctx* ctx, size_t n, const pbh_witness_record* rec, uint8_t* wit, size_t wit_pitch,
                                      uint8_t* rand, size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u);
int pbh_proof_records_to_planes_dev(pbh_ctx* ctx, size_t n, const pbh_proof_record* rec, uint8_t* proof, size_t proof_pitch,
                                    uint8_t* status);
int pbh_proof_planes_to_records_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status,
                                    pbh_proof_record* rec);

/* ---- packed wire format: the PCIe-lean form of the same batches -----------------------------------------------------------
 * Byte planes cost 59 bytes up and 29 bytes down per proof + verification, and for host-resident batches the host link, not
 * the GPU, is the bound.  Packed records carry the same values in radix form, 32 bytes up and 13 bytes down:
 *   pbh_packed_witness  16 bytes: the 27 values wit[0..12) rand[0..9) chal[0..5) u, each < 17, as base-17 digits, least
 *                       significant first: values 0..6 in w[0], 7..13 in w[1], 14..20 in w[2], 21..26 in w[3].
 *   pbh_packed_proof    12 bytes.  points (lo | hi << 32): nine base-102 digits, least significant first, one POINT CODE per
 *                       commitment in proof order.  Code 0 is the identity (0, 0, infinite); code c >= 1 is the c-th finite
 *                       point of y^2 = x^3 + 3 over F_101 in increasing (x, y) order (the curve has exactly 101 of them, so every
 *                       point a prover emits has a code; (1, 2), the generator of src/pbh/g1.rs:91-96, is code 1).  evals_status:
 *                       bits 0..28 the seven evaluations as base-17 digits, bits 29..31 the STATUS CODE: 0..5 = PBH_ST_OK ..
 *                       PBH_ST_SRS_OOB, 7 = PBH_ST_BAD_ENCODING, 6 = PBH_ST_UNREPRESENTABLE (set only when packing a proof the
 *                       format cannot express: a point off the curve, a flagged identity with coordinates, an evaluation >= 17).
 *                       Both payload words are zero whenever the status code is not 0.
 *   chal_u              4 bytes per verification: alpha beta gamma z v u as six base-17 digits.
 * PARITY UNPINNED BY THE REFERENCE as a format (the reference has no serialisation: src/plonk.rs:61); pinned by an independent
 * restatement of this text (oracle/oracle.py packed_*, tests/test_packed_format.py).  The CONTENT is pinned: semantics are
 * those of the byte-plane entry points on the decoded values, bit for bit: pbh_prove_packed(in) = pack(
 * pbh_prove_batch(unpack(in))), pbh_verify_packed(proofs, chal_u) = pbh_verify_batch(unpack(proofs), unpack(chal_u)).  A word
 * outside the format decodes to a byte outside the field (its top digit saturates at 255), hence PBH_ST_BAD_ENCODING /
 * PBH_VR_BAD_ENCODING / PBH_VR_NOT_IN_FIELD as for byte planes; a packed proof whose status code is not 0 decodes to the all-zero
 * proof that pbh_prove_batch leaves for such an item (the verifier answers PBH_VR_NOT_ON_CURVE), as does a ninth point digit
 * >= 102.  Off-curve and malformed proofs - the verifier's adversarial inputs - have no packed form: use the byte planes. */
typedef struct pbh_packed_witness { uint32_t w[4]; } pbh_packed_witness;
typedef struct pbh_packed_proof { uint32_t points_lo, points_hi, evals_status; } pbh_packed_proof;
/* Plonk::prove / Plonk::verify over packed records, HOST pointers (any memory; page-locked memory overlaps best). */
int pbh_prove_packed(pbh_ctx* ctx, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out);
int pbh_verify_packed(pbh_ctx* ctx, size_t n, const pbh_packed_proof* proofs, const uint32_t* chal_u, uint8_t* result);
/* The same on a lane (see "lanes" above): page-locked buffers are moved whole by the copy engines on the lane's stream and the
 * call returns at once; with pageable memory the call waits for the context's earlier work and runs synchronously. */
int pbh_prove_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out);
int pbh_verify_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_proof* proofs, const uint32_t* chal_u, uint8_t* result);
/* Extension: prove, then verify the fresh proofs with the same record's challenges and u; the proof never re-crosses PCIe. */
int pbh_prove_verify_packed(pbh_ctx* ctx, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out, uint8_t* result);
int pbh_prove_verify_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out, uint8_t* result);
/* Device-side conversions between packed records and byte planes (device pointers; null plane pointers are skipped). */
int pbh_unpack_witness_dev(pbh_ctx* ctx, size_t n, const pbh_packed_witness* in, uint8_t* wit, size_t wit_pitch, uint8_t* rand,
                           size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u);
int pbh_pack_proof_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status, pbh_packed_proof* out);
int pbh_unpack_proof_dev(pbh_ctx* ctx, size_t n, const pbh_packed_proof* in, const uint32_t* chal_u, uint8_t* proof, size_t proof_pitch,
                         uint8_t* status, uint8_t* chal, size_t chal_pitch, uint8_t* u);
/* Host-side format conversion (plain CPU loops over host memory; no context, no device, nothing is proved or verified): what
 * a host program uses to build packed records from its own values and to read proofs back.  pack functions return
 * PBH_ERR_BAD_ARGUMENT when a value is >= 17 (witness, chal_u); pbh_pack_proofs_host marks inexpressible proofs with status
 * code 6 instead.  Null plane pointers are skipped by the unpack functions; u / chal may be null for pbh_pack_witness_host
 * (packed as zero). */
int pbh_pack_witness_host(size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand, size_t rand_pitch, const uint8_t* chal,
                          size_t chal_pitch, const uint8_t* u, pbh_packed_witness* out);
int pbh_unpack_witness_host(size_t n, const pbh_packed_witness* in, uint8_t* wit, size_t wit_pitch, uint8_t* rand, size_t rand_pitch,
                            uint8_t* chal, size_t chal_pitch, uint8_t* u);
int pbh_pack_chal_u_host(size_t n, const uint8_t* chal, size_t chal_pitch, const uint8_t* u, uint32_t* out);
int pbh_pack_proofs_host(size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status, pbh_packed_proof* out);
int pbh_unpack_proofs_host(size_t n, const pbh_packed_proof* in, uint8_t* proof, size_t proof_pitch, uint8_t* status);

/* ---- Fiat-Shamir over packed records: the two sections above combined ------------------------------------------------------
 * A Fiat-Shamir prover takes no challenges and a Fiat-Shamir verifier takes only the proof, so the packed form of this family is
 * 12 bytes up and 12 (+4) bytes down per proof, 12 bytes up and 1 byte down per verification:
 *   pbh_packed_fs_witness  12 bytes: the 21 values wit[0..12) rand[0..9), each < 17, as base-17 digits, least significant first:
 *                          values 0..6 in w[0], 7..13 in w[1], 14..20 in w[2] - word for word words 0..2 of pbh_packed_witness.
 *                          Decoding is that of pbh_packed_witness: whatever lies above a word's seventh digit is folded into it
 *                          and saturates at 255, so a word >= 17^7 decodes to a byte >= 17 and the item gets PBH_ST_BAD_ENCODING.
 *   pbh_packed_proof       as above.
 *   chal_u_out (nullable)  4 bytes per proof: the derived alpha beta gamma z v u as the chal_u word of pbh_verify_packed (six
 *                          base-17 digits); zero where the status is not PBH_ST_OK, as chal_out of pbh_prove_fs_batch.  When it is
 *                          null the prover skips the transcript step that derives u.
 * PARITY UNPINNED BY THE REFERENCE, as both sections this one combines.  Definitions, bit for bit:
 *   pbh_prove_fs_packed(in) = pack(pbh_prove_fs_batch(unpack(in))), with chal_u_out = pack_chal_u(chal_out);
 *   pbh_verify_fs_packed(p) = pbh_verify_fs_batch(unpack(p)).
 * A packed proof whose status code is not 0 decodes to the all-zero proof and is verified as such (PBH_VR_NOT_ON_CURVE).
 * The kernels decode and encode in registers: there is no plane round trip and no extra launch.  Device record pointers must be
 * 4-byte aligned.  The verifier always uploads and checks the buffer it is given. */
typedef struct pbh_packed_fs_witness { uint32_t w[3]; } pbh_packed_fs_witness;
/* HOST pointers (any memory; page-locked memory overlaps best), chunked over the staging buffers */
int pbh_prove_fs_packed(pbh_ctx* ctx, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out);
int pbh_verify_fs_packed(pbh_ctx* ctx, size_t n, const pbh_packed_proof* proofs, uint8_t* result);
/* the same on a lane, with the contract of pbh_prove_packed_async (pageable memory: waits for the context, then synchronous) */
int pbh_prove_fs_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out,
                              uint32_t* chal_u_out);
int pbh_verify_fs_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_proof* proofs, uint8_t* result);
/* DEVICE pointers: only enqueued on the context's compute stream (may be captured into CUDA graphs) */
int pbh_prove_fs_packed_dev(pbh_ctx* ctx, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out);
int pbh_verify_fs_packed_dev(pbh_ctx* ctx, size_t n, const pbh_packed_proof* proofs, uint8_t* result);
/* host-side format conversion, as pbh_pack_witness_host / pbh_unpack_witness_host (PBH_ERR_BAD_ARGUMENT when a value is >= 17;
 * null plane pointers are skipped by the unpack function) */
int pbh_pack_fs_witness_host(size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand, size_t rand_pitch,
                             pbh_packed_fs_witness* out);
int pbh_unpack_fs_witness_host(size_t n, const pbh_packed_fs_witness* in, uint8_t* wit, size_t wit_pitch, uint8_t* rand,
                               size_t rand_pitch);

/* ---- sweep kernels (the per-kernel configs of BASELINE.json), HOST or DEVICE pointers --------- */
/* `on_device` != 0: pointers are device pointers, kernels are only enqueued.                      */

/* size-4 NTT over F_17, omega = 4: evals[i] = sum_j coeffs[j] * 4^(ij)  (src/fft.rs:66-78, 90-106
 * with EvaluationDomainGenerator(4, 4)); 4 planes in, 4 planes out. */
int pbh_ntt4_batch(pbh_ctx* ctx, size_t n, const uint8_t* coeffs, size_t in_pitch, uint8_t* evals,
                   size_t out_pitch, int on_device);
/* inverse: Plonk::interpolate_at_h (src/plonk.rs:177-179) == fft_inv (src/fft.rs:72-78), always 4
 * coefficients (zero padded; the reference's normalised length is implied by the values). */
int pbh_intt4_batch(pbh_ctx* ctx, size_t n, const uint8_t* evals, size_t in_pitch, uint8_t* coeffs,
                    size_t out_pitch, int on_device);
/* The same two transforms on a COSET k H of the order-4 subgroup: evals[i] = p(k 4^i), and its inverse.  k = 2 and k = 3 are
 * K1 and K2 of src/pbh/mod.rs:27-28, whose cosets k1_h = {2, 8, 15, 9} and k2_h = {3, 12, 14, 5} the reference builds in
 * Plonk::new (src/plonk.rs:136-139) for the copy-constraint labels; k = 1 is H itself (pbh_ntt4_batch / pbh_intt4_batch).
 * The reference has no coset transform of its own: the forward results equal Poly::eval (src/poly.rs:71-79) of the
 * polynomial at the four coset points, the inverse undoes it.  Any other k: PBH_ERR_UNSUPPORTED. */
int pbh_coset_ntt4_batch(pbh_ctx* ctx, size_t n, uint32_t k, const uint8_t* coeffs, size_t in_pitch, uint8_t* evals,
                         size_t out_pitch, int on_device);
int pbh_coset_intt4_batch(pbh_ctx* ctx, size_t n, uint32_t k, const uint8_t* evals, size_t in_pitch, uint8_t* coeffs,
                          size_t out_pitch, int on_device);
/* generic power-of-two NTT / iNTT over F_modulus (modulus < 2^16, size in {2,4,...,64}), values as
 * uint16 planes; reproduces CooleyTurkey::fft / fft_inv (src/fft.rs:66-78) for full-length input.  Inputs are reduced
 * mod modulus first; omega need not be primitive.  Only the inverse needs size^-1 mod modulus (fft_inv): without one it
 * returns PBH_ERR_SETUP_PANIC, as the reference's `inv().unwrap()` panics, while the forward transform computes (modulus 2,
 * even moduli). */
int pbh_ntt_generic_batch(pbh_ctx* ctx, size_t n, uint32_t modulus, uint32_t omega, uint32_t size, int inverse,
                          const uint16_t* in, size_t in_pitch_elems, uint16_t* out, size_t out_pitch_elems,
                          int on_device);
/* mul_ntt (src/fft.rs:109-132) with CooleyTurkey over F_modulus: a (la uint16 planes) and b (lb planes) are zero-extended
 * to la + lb values (a power of two in [2, 64], omega a primitive root of that order), transformed, multiplied
 * pointwise and transformed back; la + lb planes out (the top one is 0).  Reproduces src/fft.rs:171-183. */
int pbh_mul_ntt_batch(pbh_ctx* ctx, size_t n, uint32_t modulus, uint32_t omega, uint32_t la, uint32_t lb, const uint16_t* a,
                      size_t a_pitch_elems, const uint16_t* b, size_t b_pitch_elems, uint16_t* out, size_t out_pitch_elems,
                      int on_device);
/* The next three take `len` coefficient planes over F_17 (zero padded, len <= 64) followed by ONE operand plane.
 * Poly * scalar (src/poly.rs:220-228; the scalar plane): len planes out. */
int pbh_poly_scale_batch(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch,
                         int on_device);
/* Poly::eval at the point plane (src/poly.rs:71-79): n bytes out. */
int pbh_poly_eval_batch(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, int on_device);
/* Poly / (x - c), c the operand plane (src/poly.rs:230-247 with the linear divisors of src/plonk.rs:437-442): len planes out,
 * the len - 1 quotient coefficients then the remainder (= p(c)). */
int pbh_poly_div_linear_batch(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out,
                              size_t out_pitch, int on_device);
/* schoolbook product over F_17 (src/poly.rs:205-218): la, lb coefficient planes (zero padded) in,
 * la+lb-1 planes out (la, lb <= 16). */
int pbh_poly_mul_batch(pbh_ctx* ctx, size_t n, uint32_t la, uint32_t lb, const uint8_t* a, size_t a_pitch,
                       const uint8_t* b, size_t b_pitch, uint8_t* out, size_t out_pitch, int on_device);
/* coefficientwise a + b or a - b over F_17 on len planes (src/poly.rs:165-203 for equal lengths) */
int pbh_poly_add_batch(pbh_ctx* ctx, size_t n, uint32_t len, int subtract, const uint8_t* a, size_t a_pitch,
                       const uint8_t* b, size_t b_pitch, uint8_t* out, size_t out_pitch, int on_device);
/* (q, r) = p / (x^4 - 1) over F_17 (src/poly.rs:230-247 with rhs = Z_H, src/plonk.rs:369):
 * 22 planes in, 18 quotient planes + 4 remainder planes out. */
int pbh_poly_div_zh_batch(pbh_ctx* ctx, size_t n, const uint8_t* p, size_t p_pitch, uint8_t* q, size_t q_pitch,
                          uint8_t* r, size_t r_pitch, int on_device);
/* G1P * F101 (src/pbh/g1.rs:146-168): planes x, y, inf(0/1), k (0..100) in; x, y, inf out. */
int pbh_g1_smul_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch,
                      int on_device);
/* G1P + G1P (src/pbh/g1.rs:119-144): planes x1 y1 inf1 x2 y2 inf2 in; x y inf out.  Items for which
 * the reference would panic ("cannot add": equal x, unequal non-opposite y — unreachable for points
 * on the curve) get inf = 0xFF. */
int pbh_g1_add_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch,
                     int on_device);
/* SRS::eval_at_s (src/plonk.rs:51-58): 7 coefficient planes (F_17, zero padded) in; x, y, inf out. */
int pbh_kzg_commit_batch(pbh_ctx* ctx, size_t n, const uint8_t* coeffs, size_t in_pitch, uint8_t* out,
                         size_t out_pitch, int on_device);
/* PBHPairing::pairing (src/pbh/pairing.rs:12-47): planes p.x p.y p.inf q.a q.b in; gt.a gt.b out. */
int pbh_pairing_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch,
                      int on_device);

/* GTP * GTP (src/pbh/gt.rs:61-69): planes a1 b1 a2 b2 in; a b out.  GTP::pow(600) (src/pbh/gt.rs:33-59, the final
 * exponentiation of src/pbh/pairing.rs:17): planes a b in; a b out (0 + 0u stays 0 + 0u, Q10). */
int pbh_gt_mul_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device);
int pbh_gt_pow600_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device);
/* (q, r) = num / den for ANY divisor over F_17 (src/poly.rs:230-247): ln numerator planes and ld divisor planes in (zero
 * padded, 1 <= ln <= 32, 1 <= ld <= 16), ln quotient planes and ld remainder planes out.  status[i] = 1 where the reference
 * panics (a NON-ZERO numerator divided by the zero polynomial: `lead_d.inv().unwrap()`; 0 / 0 is (0, 0) because the division
 * loop never starts), with zero outputs; 0 otherwise. */
int pbh_poly_divrem_batch(pbh_ctx* ctx, size_t n, uint32_t ln, uint32_t ld, const uint8_t* num, size_t num_pitch, const uint8_t* den,
                          size_t den_pitch, uint8_t* q, size_t q_pitch, uint8_t* r, size_t r_pitch, uint8_t* status, int on_device);
/* `a += b` (subtract = 0) / `a -= b` (subtract = 1) for operands of different lengths exactly as the reference does it
 * (src/poly.rs:165-176, 192-203): la and lb planes in (zero padded, <= 64), max(la, lb) planes out.  With len(a) the
 * normalised length of a, out[n] = a[n] +- b[n] below len(a) and b[n] UNCHANGED at or beyond it - also when subtracting,
 * which is the quirk (SURVEY.md Q1) the prover depends on. */
int pbh_poly_addsub_ragged_batch(pbh_ctx* ctx, size_t n, uint32_t la, uint32_t lb, int subtract, const uint8_t* a, size_t a_pitch,
                                 const uint8_t* b, size_t b_pitch, uint8_t* out, size_t out_pitch, int on_device);

/* ---- shard summaries for the multi-GPU gather (SURVEY.md §8e) ---------------------------------- */
/* Pack bit 0 of each result byte into a bitmap (item i -> bit i%8 of byte i/8), device pointers.  */
int pbh_pack_verdicts_dev(pbh_ctx* ctx, size_t n, const uint8_t* result, uint8_t* bitmap);
/* 64-bit digest of `planes` byte planes of n items starting at global item index `first_index`.  Per item: the bytes
 * are packed four planes per little-endian 32-bit word and mixed into two 32-bit lanes seeded with the global index
 * (murmur3-style multiply/rotate rounds, murmur3 finaliser); the batch digest is the sum of the 64-bit item values
 * modulo 2^64, so digests of disjoint shards add up to the digest of the whole batch.  out: one uint64 (device). */
int pbh_digest_dev(pbh_ctx* ctx, size_t n, uint64_t first_index, uint32_t planes, const uint8_t* data, size_t pitch,
                   uint64_t* out);

/* Fused variants for the multi-GPU summaries (device pointers).  Same results as the plain entry points followed by
 * pbh_digest_dev(proof) / pbh_pack_verdicts_dev(result); the prover adds the digest of its 27 proof planes while the
 * bytes are still in registers and the verifier packs the verdict bits with a warp ballot.
 *   digest: one uint64, overwritten; bitmap: ceil(n/8) bytes, 4-byte aligned. */
int pbh_prove_digest_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand,
                               size_t rand_pitch, const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch,
                               uint8_t* status, uint64_t first_index, uint64_t* digest);
int pbh_verify_bitmap_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                                size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* bitmap);
/* The same for the Fiat-Shamir calls: pbh_prove_fs_batch_dev followed by pbh_digest_dev(27 proof planes, first_index), and
 * pbh_verify_fs_batch_dev followed by pbh_pack_verdicts_dev(result).  chal_out (nullable) as in pbh_prove_fs_batch_dev.  The
 * FP32 provers add the digest in the kernel; with PBH_OPT_PROVER_FP32 = 0 the digest kernel runs after the prover.  A bitmap
 * that is not 4-byte aligned is packed by a second kernel.  Both take part in peer windows like the two calls above. */
int pbh_prove_fs_digest_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand,
                                  size_t rand_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out,
                                  size_t chal_pitch, uint64_t first_index, uint64_t* digest);
int pbh_verify_fs_bitmap_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result,
                                   uint8_t* bitmap);

/* ---- peer windows: the gather of the shard summaries as plain stores over NVLink ----------------------------------------
 * The only exchange of the sharded path is that every device ends up with every shard's verdict bitmap and proof digest
 * (SURVEY.md 8e).  A collective after the kernels costs a rendezvous per call; a peer window removes it: every rank owns a
 * device buffer of world x bytes_per_rank bytes, rank r's region being bytes [r * bytes_per_rank, (r + 1) * bytes_per_rank)
 * of EVERY rank's buffer.  When the `digest` of pbh_prove_digest_batch_dev / pbh_prove_fs_digest_batch_dev or the `bitmap` of
 * pbh_verify_bitmap_batch_dev / pbh_verify_fs_bitmap_batch_dev points into the calling rank's own region, the kernel that produces the summary also stores it at the same offset of every
 * peer's buffer - the verifier per 256-item tile (one 32-byte store per peer), the prover's last block its 8-byte digest -
 * through peer-mapped device memory (NVLink / NVSwitch), so the all-gather has happened when the kernels have finished and
 * costs neither a launch nor a rendezvous.  A consumer on another rank must be ordered after the producing rank's stream
 * (a barrier at the end of a pass).  world <= 8; bytes_per_rank a multiple of 16.
 *   pbh_window_create      allocates (zeroed) this rank's buffer; base_out = its device address; handle_out (nullable) = a
 *                          CUDA IPC handle other PROCESSES open with pbh_window_attach (one process per GPU, torchrun)
 *   pbh_window_attach      handles: world x PBH_IPC_HANDLE_BYTES bytes, entry r from rank r (the own entry is ignored)
 *   pbh_window_attach_ptrs the same for peers of THIS process: their buffers' device addresses (peer access is enabled)
 *   pbh_window_share       lets another context of the same device (its own stream) write through an attached window
 *   pbh_window_destroy     detaches and frees; also done by pbh_ctx_destroy */
#define PBH_IPC_HANDLE_BYTES 64
int pbh_window_create(pbh_ctx* ctx, size_t bytes_per_rank, int rank, int world, void** base_out, uint8_t handle_out[PBH_IPC_HANDLE_BYTES]);
int pbh_window_attach(pbh_ctx* ctx, const uint8_t* handles);
int pbh_window_attach_ptrs(pbh_ctx* ctx, void* const* bases);
int pbh_window_share(pbh_ctx* owner, pbh_ctx* other);
int pbh_window_destroy(pbh_ctx* ctx);

/* ---- multi-device: several GPUs driven from ONE process (SURVEY.md §8b, §8e) -------------------------------------------
 * pbh_multi_create does pbh_ctx_create on each of the n_dev devices (devices == NULL: 0 .. n_dev-1), with one stream per
 * device, and - when n_dev > 1 - builds one NCCL communicator over them (ncclCommInitAll; libnccl.so.2 is loaded at run
 * time, PBH_ERR_UNSUPPORTED when it cannot be: there is no fallback for the collective).  Batches are split contiguously
 * over the devices in whole 256-item tiles.  Results never depend on the number of devices.  (The one-process-per-GPU
 * arrangement under torchrun uses plain contexts and torch.distributed instead: plonk-by-fingers_b200/python/pbh_b200/
 * sharding.py, bench.py.) */
typedef struct pbh_multi pbh_multi;
int pbh_multi_create(const pbh_circuit* circuit, uint8_t srs_secret, uint32_t srs_n, uint8_t omega_pows, const int* devices,
                     int n_dev, pbh_multi** out);
void pbh_multi_destroy(pbh_multi* m);
int pbh_multi_device_count(const pbh_multi* m);
pbh_ctx* pbh_multi_ctx(pbh_multi* m, int i);              /* the context of device i, e.g. for the `_dev` entry points */
const char* pbh_multi_last_error(const pbh_multi* m);     /* m may be NULL: last creation error */
int pbh_multi_set_algo(pbh_multi* m, int algo);
/* Plonk::prove / Plonk::verify over n items, HOST pointers, same arguments and bytes as pbh_prove_batch / pbh_verify_batch:
 * shard d goes through device d's single-device entry point on its own host thread. */
int pbh_multi_prove_batch(pbh_multi* m, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand, size_t rand_pitch,
                          const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status);
int pbh_multi_verify_batch(pbh_multi* m, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                           size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch);
/* The same over packed records (pbh_prove_packed / pbh_verify_packed per shard). */
int pbh_multi_prove_packed(pbh_multi* m, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out);
int pbh_multi_verify_packed(pbh_multi* m, size_t n, const pbh_packed_proof* proofs, const uint32_t* chal_u, uint8_t* result);
/* The sharded end-to-end pass of BASELINE.json configs[4] in one call.  The synthetic items with global indices
 * [first_index, first_index + n_total) (pbh_generate_inputs_dev) are generated, proved and verified shard by shard on the
 * devices, the digest fused into the prover and the verdict bitmap into the verifier; then ONE ncclAllGather exchanges the
 * shard summaries (bitmap + 64-bit proof digest), after which every device holds all of them.  Returned from device 0:
 *   bitmap_out        ceil(n_total / 8) bytes, bit i%8 of byte i/8 = verdict of item i (what one device computes alone)
 *   digests_out       n_dev values (nullable); total_digest_out (nullable) their sum mod 2^64 = pbh_digest_dev of the whole batch
 *   accepted_out      number of accepted proofs (nullable)
 *   ms_out            device time of the pass including the collective, maximum over the devices, CUDA events (nullable) */
int pbh_multi_prove_verify_sharded(pbh_multi* m, uint64_t n_total, uint64_t first_index, uint64_t seed, int dist,
                                   uint8_t* bitmap_out, uint64_t* digests_out, uint64_t* total_digest_out, uint64_t* accepted_out,
                                   float* ms_out);
/* Fiat-Shamir over several devices, host pointers: same arguments and bytes as pbh_prove_fs_batch / pbh_verify_fs_batch /
 * pbh_prove_fs_packed / pbh_verify_fs_packed, shard d through device d's entry point on its own host thread. */
int pbh_multi_prove_fs_batch(pbh_multi* m, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rand, size_t rand_pitch,
                             uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch);
int pbh_multi_verify_fs_batch(pbh_multi* m, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result,
                              uint8_t* chal_out, size_t chal_pitch, uint8_t* gt, size_t gt_pitch);
int pbh_multi_prove_fs_packed(pbh_multi* m, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out);
int pbh_multi_verify_fs_packed(pbh_multi* m, size_t n, const pbh_packed_proof* proofs, uint8_t* result);
/* pbh_multi_prove_verify_sharded with the Fiat-Shamir transcript: per shard pbh_generate_inputs_dev (its challenge and u planes
 * are not used), pbh_prove_fs_digest_batch_dev (chal_out = NULL), pbh_verify_fs_bitmap_batch_dev, then the same all-gather.
 * Outputs as there; bitmap_out and the digests equal what one device computes alone for the same global index range. */
int pbh_multi_prove_verify_fs_sharded(pbh_multi* m, uint64_t n_total, uint64_t first_index, uint64_t seed, int dist,
                                      uint8_t* bitmap_out, uint64_t* digests_out, uint64_t* total_digest_out,
                                      uint64_t* accepted_out, float* ms_out);

/* ---- synthetic inputs (SURVEY.md §8d), device pointers ------------------------------------------ */
#define PBH_DIST_UNIFORM 0   /* attempt k = 0 only: exercises every status class                    */
#define PBH_DIST_FULLPATH 1  /* smallest k whose prove succeeds and whose verify reaches the pairing */
/* The full-path search tries attempts k = 0 .. PBH_GEN_MAX_ATTEMPTS - 1.  An item none of them satisfies (a short SRS
 * where every proof ends in PBH_ST_SRS_OOB or commits to the identity) gets attempt 0's draw with attempt byte 255.  On
 * the reference's circuit and SRS an attempt succeeds with probability about 1/19, so the cap is never reached there.  Witnesses are drawn
 * from the 289 solutions (x, y, z) of x^2 + y^2 = z^2 (wit = x y z x^2, x y z y^2, x^2 y^2 z^2 z^2); on a context whose
 * gates and copy constraints no such row satisfies, PBH_DIST_FULLPATH returns PBH_ERR_UNSUPPORTED before any launch. */
#define PBH_GEN_MAX_ATTEMPTS 4096
/* Item i of the batch has global index first_index + i; its bytes depend only on (seed, global
 * index, dist), so any sharding generates the same batch.  Fills wit/rand/chal/u; `attempt`
 * (nullable, n bytes) receives the accepted k (saturating at 255). */
int pbh_generate_inputs_dev(pbh_ctx* ctx, size_t n, uint64_t first_index, uint64_t seed, int dist, uint8_t* wit,
                            size_t wit_pitch, uint8_t* rand, size_t rand_pitch, uint8_t* chal, size_t chal_pitch,
                            uint8_t* u, uint8_t* attempt);

/* ---- measurement helpers ------------------------------------------------------------------------ */
/* Pipe-rate micro-benchmark (independent register chains, no memory traffic): thread-level operations per second
 * the device sustains for one instruction class; the INT32 / FMA roofline denominators of SURVEY.md §8d.
 * which: 0 IMAD, 1 LOP3+IADD3, 2 half IMAD half ALU, 3 FFMA, 4 HFMA2 (counted once per instruction; each carries two
 * fp16 lanes), 5 IDP.4A (dp4a; four byte MACs each), 6 IMAD.HI+IADD, 7 half FFMA half IMAD,
 * 8 FFMA with three register operands (polynomial MAC shape), 9 IMAD with three register operands,
 * 10 FFMA2 (packed fp32x2, counted per instruction) with three register-pair operands, 11 FFMA2 with a broadcast-pair multiplicand,
 * 12 SHF (funnel shift), 13 IMAD.WIDE.U32, 14 LOP3 alone, 15 IADD3 alone, 16 PRMT (the SHA-256 transcript's instruction classes) */
int pbh_measure_int32_peak(pbh_ctx* ctx, int which, double* lane_ops_per_second);

#ifdef __cplusplus
}
#endif
#endif /* PBH_B200_H */
