// pbh_kernels.cuh — sm_100a kernels: fused prover, fused verifier, the sweep kernels of BASELINE.json,
// the synthetic-input generator, shard summaries and the INT32 peak micro-benchmark.
//
// Layout: structure-of-arrays byte planes (include/pbh_b200.h).  One thread handles one item per
// grid-stride step; consecutive threads touch consecutive bytes of every plane, so each warp-wide load or
// store is one fully used 32-byte sector.  Grids are sized as a multiple of the SM count and blocks stage the
// context's lookup tables (~2.7 KB) into shared memory once, then loop.  No tensor cores: nothing on this
// path is a dense contraction.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "../../include/pbh_b200.h"
#include "pbh_verify.cuh"
#include "pbh_prove_f32.cuh"
#include "pbh_tma.cuh"
#include "pbh_packed.cuh"

namespace pbh {

constexpr int kBlock = 256;

__device__ __forceinline__ void stage_tables(Tables& sT, const Tables* __restrict__ gT) {
  const uint32_t* src = reinterpret_cast<const uint32_t*>(gT);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&sT);
  for (int i = threadIdx.x; i < (int)(sizeof(Tables) / 4); i += blockDim.x) dst[i] = src[i];
  __syncthreads();
}

// Digest of one item (include/pbh_b200.h): two 32-bit lanes, murmur3-style rounds over the item's bytes packed four
// planes per word, murmur3 finaliser.  32-bit multiplies only: cheap on the integer pipes.
struct DigestState { uint32_t a, b; };
__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return __funnelshift_l(x, x, r); }
__device__ __forceinline__ uint32_t fmix32(uint32_t h) { h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16; return h; }
__device__ __forceinline__ DigestState digest_item_begin(uint64_t index, uint32_t planes) {
  DigestState d;
  d.a = (uint32_t)index * 0x9E3779B1u + planes;
  d.b = (uint32_t)(index >> 32) * 0x85EBCA77u + 0x27D4EB2Fu;
  return d;
}
__device__ __forceinline__ void digest_item_word(DigestState& d, uint32_t wv) {
  d.a = rotl32((d.a ^ wv) * 0xCC9E2D51u, 15);
  d.b = rotl32((d.b + wv) * 0x1B873593u, 13) ^ d.a;
}
__device__ __forceinline__ unsigned long long digest_item_end(const DigestState& d) {
  return ((unsigned long long)fmix32(d.a ^ rotl32(d.b, 16)) << 32) | fmix32(d.b + d.a);
}
// warp-reduce and add a per-thread partial sum into *out (one atomic per warp)
__device__ __forceinline__ void digest_flush(unsigned long long acc, unsigned long long* out) {
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

// Dynamic tile scheduler state: c[0] = next tile, c[1] = blocks finished (c[2..3]: the prover's 64-bit digest accumulator).  The record is launch-local (the host hands every
// launch its own, pbh_capi.cu: fresh_tile_counter) and zero when the launch starts: the last block to leave resets it, so
// a launch recorded into a CUDA graph finds it zero again at every replay and no memset node is needed.
// Returns true in thread 0 of the LAST block to leave (every other block's writes that preceded its own leave are then visible
// to that thread).
__device__ __forceinline__ bool tile_scheduler_leave(unsigned int* c) {
  bool last = false;
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&c[1], 1u) == gridDim.x - 1) {
      c[0] = 0u;
      c[1] = 0u;
      __threadfence();
      last = true;
    }
  }
  return last;
}

// Peer window (include/pbh_b200.h "peer windows"): the shard summaries a kernel writes (the verifier's verdict bitmap, the
// prover's proof digest) are ALSO stored, by the same kernel, at the same offset of every peer's window - plain stores over
// NVLink into peer memory - so that after the kernel every device holds this shard's summary and no collective is needed.
struct PeerWindow {
  uint32_t n;            // number of peers (0: not replicated)
  long long delta[7];    // peer address = local address + delta[p]
};

// Digest of one item's 27 proof bytes as store_proof writes them (pbh_digest_dev's definition), from registers: planes
// 4k..4k+3 per word.  pp: the nine point words' low 16 bits, ee: the seven evaluations, all zero when the status is not 0.
__device__ __forceinline__ unsigned long long proof_item_digest(uint64_t index, const uint32_t (&pp)[9], uint32_t inf_lo, uint32_t inf_hi,
                                                                const uint32_t (&ee)[7]) {
  DigestState d = digest_item_begin(index, 27);
  digest_item_word(d, pp[0] | (pp[1] << 16));
  digest_item_word(d, pp[2] | (pp[3] << 16));
  digest_item_word(d, pp[4] | (pp[5] << 16));
  digest_item_word(d, pp[6] | (pp[7] << 16));
  digest_item_word(d, pp[8] | (inf_lo << 16) | (inf_hi << 24));
  digest_item_word(d, ee[0] | (ee[1] << 8) | (ee[2] << 16) | (ee[3] << 24));
  digest_item_word(d, ee[4] | (ee[5] << 8) | (ee[6] << 16));
  return digest_item_end(d);
}

// A prover's per-thread digest sums -> ONE atomic per block into the launch-local accumulator next to the tile counters
// (c[2..3], zero when the launch starts, like them): no memset of the digest word is needed in front of the kernel.  2368
// same-address atomics (one per warp) at the end of a 2^20-item launch serialise in L2 for microseconds; 296 do not.
// part: kBlock / 32 words of shared memory.  Ends with the block barrier tile_scheduler_leave relies on.
__device__ __forceinline__ void digest_block_add(unsigned long long acc, unsigned long long* part, unsigned int* c) {
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long sum = 0;
#pragma unroll
    for (int k = 0; k < kBlock / 32; k++) sum += part[k];
    atomicAdd(reinterpret_cast<unsigned long long*>(c + 2), sum);
  }
}
// Thread 0 of the last block to leave (tile_scheduler_leave; every block's digest atomic precedes the fence there): every block
// has added its share, so it publishes the launch's digest (overwriting *digest_out), re-arms the accumulator for the next launch
// that is handed this record, and pushes the digest to every peer's window.
__device__ __forceinline__ void digest_publish(unsigned int* c, unsigned long long* digest_out, const PeerWindow& PW) {
  __threadfence();
  volatile unsigned long long* acc = reinterpret_cast<volatile unsigned long long*>(c + 2);
  const unsigned long long d = *acc;
  *acc = 0ull;
  *digest_out = d;
#pragma unroll
  for (uint32_t p = 0; p < 7; p++)     // fixed trip count: delta[] stays in the parameter bank (no local copy)
    if (p < PW.n) *reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(digest_out) + PW.delta[p]) = d;
  __threadfence();
}

struct ProveArgs {
  const uint8_t* wit; size_t wit_pitch;
  const uint8_t* rnd; size_t rand_pitch;
  const uint8_t* chal; size_t chal_pitch;
  uint8_t* proof; size_t proof_pitch;
  uint8_t* status;
  size_t n;
};

__device__ __forceinline__ void store_proof(const ProveArgs& A, size_t i, const ProofRegs& P, uint32_t status) {
  uint32_t inf_lo = 0, inf_hi = 0;
  const bool ok = status == 0u;
#pragma unroll
  for (int k = 0; k < 9; k++) {
    uint32_t w = ok ? P.pt[k] : 0u;
    A.proof[(size_t)(2 * k) * A.proof_pitch + i] = (uint8_t)(w & 0xFF);
    A.proof[(size_t)(2 * k + 1) * A.proof_pitch + i] = (uint8_t)((w >> 8) & 0xFF);
    uint32_t inf = (w >> 16) & 1u;
    if (k < 8) inf_lo |= inf << k; else inf_hi |= inf;
  }
  A.proof[(size_t)18 * A.proof_pitch + i] = (uint8_t)inf_lo;
  A.proof[(size_t)19 * A.proof_pitch + i] = (uint8_t)inf_hi;
#pragma unroll
  for (int k = 0; k < 7; k++) A.proof[(size_t)(20 + k) * A.proof_pitch + i] = (uint8_t)(ok ? P.ev[k] : 0u);
  A.status[i] = (uint8_t)status;
}

// Plonk::prove, src/plonk.rs:191-466
template <int ALGO>
__global__ void __launch_bounds__(kBlock) prove_kernel(const Consts K, const Tables* __restrict__ gT, const ProveArgs A) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t w[12], r[9], c[5];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 12; k++) { w[k] = A.wit[(size_t)k * A.wit_pitch + i]; bad = bad || w[k] >= 17u; }
#pragma unroll
    for (int k = 0; k < 9; k++) { r[k] = A.rnd[(size_t)k * A.rand_pitch + i]; bad = bad || r[k] >= 17u; }
#pragma unroll
    for (int k = 0; k < 5; k++) { c[k] = A.chal[(size_t)k * A.chal_pitch + i]; bad = bad || c[k] >= 17u; }
    if (bad) {
#pragma unroll
      for (int k = 0; k < 12; k++) w[k] = 0;
#pragma unroll
      for (int k = 0; k < 9; k++) r[k] = 0;
#pragma unroll
      for (int k = 0; k < 5; k++) c[k] = 0;
    }
    ProofRegs P;
    uint32_t status = prove_one<ALGO>(w, r, c, K, sT, P);
    if (bad) status = PBH_ST_BAD_ENCODING;
    store_proof(A, i, P, status);
  }
}

// Plonk::prove with the F_17 arithmetic on the FP32 FMA pipes (pbh_prove_f32.cuh); PBH_ALGO_TABLE only
template <int ALGO, int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) prove_f32_kernel(const Consts K, const ConstsF KF, const Tables* __restrict__ gT,
                                                                         const ProveArgs A) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t w[12], r[9], c[5];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 12; k++) { w[k] = A.wit[(size_t)k * A.wit_pitch + i]; bad = bad || w[k] >= 17u; }
#pragma unroll
    for (int k = 0; k < 9; k++) { r[k] = A.rnd[(size_t)k * A.rand_pitch + i]; bad = bad || r[k] >= 17u; }
#pragma unroll
    for (int k = 0; k < 5; k++) { c[k] = A.chal[(size_t)k * A.chal_pitch + i]; bad = bad || c[k] >= 17u; }
    if (bad) {
#pragma unroll
      for (int k = 0; k < 12; k++) w[k] = 0;
#pragma unroll
      for (int k = 0; k < 9; k++) r[k] = 0;
#pragma unroll
      for (int k = 0; k < 5; k++) c[k] = 0;
    }
    ProofRegs P;
    uint32_t status = prove_item_f32<ALGO>(w, r, c, K, KF, sT, P);
    if (bad) status = PBH_ST_BAD_ENCODING;
    store_proof(A, i, P, status);
  }
}

// ---- Fiat-Shamir prover (SURVEY.md §8(f) row 1): no challenge planes in; five SHA-256 compressions per proof make the
// kernel ALU-bound (integer pipes), so it keeps plain per-thread loads and stores.
struct FsSeed { uint32_t w[8]; };
struct ProveFsArgs {
  ProveArgs base;                        // chal unused
  uint8_t* chal_out; size_t chal_pitch;  // nullable: 6 planes alpha beta gamma z v u (zero when status != 0)
};
// DIGEST instantiation only: the launch's proof digest, by the mechanism of prove_f32_tma_kernel
struct FsDigestArgs {
  uint64_t first_index;                  // global index of item 0
  unsigned long long* digest;            // overwritten by the last block to leave
  unsigned int* tile_counter;            // the launch-local record (pbh_capi.cu fresh_tile_counter): c[1] and c[2..3] are used
  PeerWindow PW;
};
// DIGEST: a compile-time flag, not a run-time branch, so that the plain instantiations compile as they did (see verify_tma_kernel).
template <int ALGO, bool FP32, bool PBH_CIRCUIT, bool DIGEST = false>
__global__ void __launch_bounds__(256, 2) prove_fs_kernel(const Consts K, const ConstsF KF, const FsSeed seed, const Tables* __restrict__ gT,
                                                           const ProveFsArgs F, const FsDigestArgs D) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  const ProveArgs& A = F.base;
  // DIGEST: the thread's running sum lives in shared memory and its slot is found from %tid.x where it is used, so that no
  // register is held across the item loop for it.  The FP32 provers use all 128 registers two resident blocks allow: with a
  // register sum the ARITH and generic TABLE instantiations spilled 56 and 32 bytes, with this 44 and 8.
  __shared__ unsigned long long digest_acc[DIGEST ? 256 : 1];
  if constexpr (DIGEST) digest_acc[threadIdx.x] = 0;
  auto slot = [&]() -> unsigned long long& { uint32_t t; asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t)); return digest_acc[t]; };
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t w[12], r[9];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 12; k++) { w[k] = A.wit[(size_t)k * A.wit_pitch + i]; bad = bad || w[k] >= 17u; }
#pragma unroll
    for (int k = 0; k < 9; k++) { r[k] = A.rnd[(size_t)k * A.rand_pitch + i]; bad = bad || r[k] >= 17u; }
    if (bad) {
#pragma unroll
      for (int k = 0; k < 12; k++) w[k] = 0;
#pragma unroll
      for (int k = 0; k < 9; k++) r[k] = 0;
    }
    ProofRegs P;
    uint32_t derived[6];
    uint32_t status = prove_item_fs<ALGO, FP32, PBH_CIRCUIT>(w, r, seed.w, K, KF, sT, P, derived, F.chal_out != nullptr);
    if (bad) status = PBH_ST_BAD_ENCODING;
    store_proof(A, i, P, status);
    if (F.chal_out) {
#pragma unroll
      for (int k = 0; k < 6; k++) F.chal_out[(size_t)k * F.chal_pitch + i] = (uint8_t)(status == 0u ? derived[k] : 0u);
    }
    if constexpr (DIGEST) {
      const bool ok = status == 0u;
      uint32_t pp[9], ee[7], inf_lo = 0, inf_hi = 0;
#pragma unroll
      for (int k = 0; k < 9; k++) {
        const uint32_t pw = ok ? P.pt[k] : 0u;
        pp[k] = pw & 0xFFFFu;
        const uint32_t inf = (pw >> 16) & 1u;
        if (k < 8) inf_lo |= inf << k; else inf_hi |= inf;
      }
#pragma unroll
      for (int k = 0; k < 7; k++) ee[k] = ok ? P.ev[k] : 0u;
      slot() += proof_item_digest(D.first_index + i, pp, inf_lo, inf_hi, ee);
    }
  }
  if constexpr (DIGEST) {
    __shared__ unsigned long long part[kBlock / 32];
    digest_block_add(digest_acc[threadIdx.x], part, D.tile_counter);
    if (tile_scheduler_leave(D.tile_counter)) digest_publish(D.tile_counter, D.digest, D.PW);
  }
}

// ---- TMA-staged prover -------------------------------------------------------------------------------------------
// Persistent blocks walk 256-item tiles.  One elected thread issues three TMA tile loads (witness, blinder and
// challenge planes) for tile k+1 into the other shared-memory stage while the block computes tile k; completion is an
// mbarrier transaction count.  Each thread then reads its 26 bytes with immediate-offset LDS (no per-plane address
// arithmetic), the copy-constraint partner of a witness value is one LDS at a uniform offset, and the 27 proof planes
// leave through one TMA tile store per tile (double-buffered; the hardware clips the ragged last tile).
constexpr int kTile = 256;
struct ProveTmaMaps {
  CUtensorMap wit, rnd, chal, proof;   // 2-D u8 tensors (n items, planes), box = (kTile, planes)
};
struct ProveTmaSmem {
  alignas(128) uint8_t in[2][26][kTile];    // planes 0..11 witness, 12..20 blinders, 21..25 challenges
  alignas(128) uint8_t out[2][27][kTile];
  alignas(8) uint64_t full[2];
  uint32_t tile_of_stage[2];                // dynamic tile scheduler: tile index staged in each buffer
  alignas(8) unsigned long long digest_part[kTile / 32];   // per-warp digest sums, folded into ONE atomic per block
  Tables T;
};

template <int ALGO, bool PBH_CIRCUIT>
__global__ void __launch_bounds__(kTile, 2) prove_f32_tma_kernel(const __grid_constant__ ProveTmaMaps M, const Consts K, const ConstsF KF,
                                                                  const Tables* __restrict__ gT, uint8_t* __restrict__ proof_out,
                                                                  size_t proof_pitch, uint8_t* __restrict__ status_out, size_t n,
                                                                  uint64_t first_index, unsigned long long* __restrict__ digest_out,
                                                                  unsigned int* __restrict__ tile_counter, const PeerWindow PW) {
  __shared__ ProveTmaSmem S;
  unsigned long long digest_acc = 0;
  const int tid = threadIdx.x;
  const size_t tiles = (n + kTile - 1) / kTile;
  auto issue = [&](size_t tile, int stage) {
    tma::mbar_arrive_expect_tx(&S.full[stage], 26 * kTile);
    const int32_t c0 = (int32_t)(tile * kTile);
    tma::load_2d(&S.in[stage][0][0], &M.wit, &S.full[stage], c0, 0);
    tma::load_2d(&S.in[stage][12][0], &M.rnd, &S.full[stage], c0, 0);
    tma::load_2d(&S.in[stage][21][0], &M.chal, &S.full[stage], c0, 0);
  };
  // Tiles are handed out by an atomic counter (zero when the launch starts), one iteration ahead of their use so that the TMA
  // prefetch overlaps the current tile: blocks that start late, e.g. because a collective's CTAs hold an SM, simply take fewer
  // tiles, and there is no wave-quantisation tail.  The index is fetched two iterations ahead (`pending`), so the atomic's
  // round trip is never waited for.  (A static first tile - the block index, loads issued before the tables are staged - was
  // measured: nothing gained at 2^20 items, 1.4 % (TABLE) to 4.5 % (ARITH) lost at 2^24.)
  // The two atomics leave first and fly while the whole block stages the tables; their results are not needed before that.
  uint32_t pending = 0, t0 = 0;
  if (tid == 0) {
    t0 = atomicAdd(tile_counter, 1u);
    pending = atomicAdd(tile_counter, 1u);
    tma::mbar_init(&S.full[0], 1);
    tma::mbar_init(&S.full[1], 1);
    tma::fence_mbar_init();
  }
  stage_tables(S.T, gT);                                      // ends with a block barrier
  if (tid == 0) {
    S.tile_of_stage[0] = t0;
    if (t0 < tiles) issue(t0, 0);
  }
  __syncthreads();
  uint32_t phase0 = 0, phase1 = 0;
  for (int stage = 0;; stage ^= 1) {
    const size_t tile = S.tile_of_stage[stage];
    if (tile >= tiles) break;
    if (tid == 0) {                                           // the other stage was released by the barrier below
      const uint32_t nt = pending;
      S.tile_of_stage[stage ^ 1] = nt;
      if (nt < tiles) {
        issue(nt, stage ^ 1);
        pending = atomicAdd(tile_counter, 1u);                // consumed in the next iteration
      }
    }
    if (stage == 0) { tma::mbar_wait(&S.full[0], phase0); phase0 ^= 1; } else { tma::mbar_wait(&S.full[1], phase1); phase1 ^= 1; }

    const uint32_t it = (uint32_t)tid;
    const uint8_t* in = &S.in[stage][0][it];
    uint32_t w[12], r[9], c[5];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 12; k++) { w[k] = in[k * kTile]; bad = bad | (w[k] >= 17u); }
#pragma unroll
    for (int k = 0; k < 9; k++) { r[k] = in[(12 + k) * kTile]; bad = bad | (r[k] >= 17u); }
#pragma unroll
    for (int k = 0; k < 5; k++) { c[k] = in[(21 + k) * kTile]; bad = bad | (c[k] >= 17u); }
    // constraints.satisfies: gates from registers, copy-constraint partners straight from the staged tile
    bool unsat = gates_unsatisfied(w, K);
#pragma unroll
    for (int k = 0; k < 12; k++) unsat = unsat | ((uint32_t)in[K.perm[k] * kTile] != w[k]);
    if (bad) {
#pragma unroll
      for (int k = 0; k < 12; k++) w[k] = 0;
#pragma unroll
      for (int k = 0; k < 9; k++) r[k] = 0;
#pragma unroll
      for (int k = 0; k < 5; k++) c[k] = 0;
    }
    ProofRegs P;
    uint32_t status = prove_item_f32<ALGO, PBH_CIRCUIT>(w, r, c, K, KF, S.T, P, unsat ? 1 : 0);
    if (bad) status = PBH_ST_BAD_ENCODING;

    uint8_t* out = &S.out[stage][0][it];
    uint32_t inf_lo = 0, inf_hi = 0;
    const bool ok = status == 0u;
#pragma unroll
    for (int k = 0; k < 9; k++) {
      uint32_t pw = ok ? P.pt[k] : 0u;
      out[(2 * k) * kTile] = (uint8_t)pw;
      out[(2 * k + 1) * kTile] = (uint8_t)(pw >> 8);
      uint32_t inf = (pw >> 16) & 1u;
      if (k < 8) inf_lo |= inf << k; else inf_hi |= inf;
    }
    out[18 * kTile] = (uint8_t)inf_lo;
    out[19 * kTile] = (uint8_t)inf_hi;
#pragma unroll
    for (int k = 0; k < 7; k++) out[(20 + k) * kTile] = (uint8_t)(ok ? P.ev[k] : 0u);
    const size_t i = tile * kTile + it;
    if (i < n) status_out[i] = (uint8_t)status;
    if (digest_out != nullptr && i < n) {
      uint32_t pp[9], ee[7];
#pragma unroll
      for (int k = 0; k < 9; k++) pp[k] = ok ? (P.pt[k] & 0xFFFFu) : 0u;
#pragma unroll
      for (int k = 0; k < 7; k++) ee[k] = ok ? P.ev[k] : 0u;
      digest_acc += proof_item_digest(first_index + i, pp, inf_lo, inf_hi, ee);
    }

    // TMA clips the item dimension at 16-byte granularity (measured), so a partial last tile whose end is not 16-byte
    // aligned is written with plain stores instead
    const bool tma_store = (tile + 1) * kTile <= n || (n & 15) == 0;
    if (!tma_store && i < n) {
#pragma unroll
      for (int k = 0; k < 27; k++) proof_out[(size_t)k * proof_pitch + i] = out[k * kTile];
    }
    // the store issued one iteration ago (other out buffer) must have finished reading shared memory before anyone
    // writes that buffer again in the next iteration; it has had a whole tile of compute to do so
    if (tid == 0) tma::store_wait_read_all();
    tma::fence_proxy_async();          // this thread's shared-memory writes -> visible to the TMA engine
    __syncthreads();                   // also releases in[stage] for the prefetch of the iteration after next
    if (tid == 0 && tma_store) {
      tma::store_2d(&M.proof, &S.out[stage][0][0], (int32_t)(tile * kTile), 0);
      tma::store_commit();
    }
  }
  if (tid == 0) tma::store_wait_all();
  if (digest_out != nullptr) digest_block_add(digest_acc, S.digest_part, tile_counter);
  const bool last = tile_scheduler_leave(tile_counter);              // thread 0: its digest atomic precedes the fence in leave
  if (last && digest_out != nullptr) digest_publish(tile_counter, digest_out, PW);
}

struct VerifyArgs {
  const uint8_t* proof; size_t proof_pitch;
  const uint8_t* chal; size_t chal_pitch;
  const uint8_t* u;
  uint8_t* result;
  uint8_t* gt; size_t gt_pitch;   // nullable
  size_t n;
  uint8_t* bitmap;                // nullable, 4-byte aligned: verdict bit of item i -> bit i%8 of byte i/8 (TMA kernel, BITMAP verify_fs_kernel)
};

// Plonk::verify, src/plonk.rs:468-650
template <int ALGO>
__global__ void __launch_bounds__(kBlock) verify_kernel(const Consts K, const ConstsF KF, const bool fp32, const Tables* __restrict__ gT,
                                                         const VerifyArgs A) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t px[9], py[9], ev[7], ch[5];
#pragma unroll
    for (int k = 0; k < 9; k++) {
      px[k] = A.proof[(size_t)(2 * k) * A.proof_pitch + i];
      py[k] = A.proof[(size_t)(2 * k + 1) * A.proof_pitch + i];
    }
    uint32_t infbits = (uint32_t)A.proof[(size_t)18 * A.proof_pitch + i] | ((uint32_t)A.proof[(size_t)19 * A.proof_pitch + i] << 8);
#pragma unroll
    for (int k = 0; k < 7; k++) ev[k] = A.proof[(size_t)(20 + k) * A.proof_pitch + i];
#pragma unroll
    for (int k = 0; k < 5; k++) ch[k] = A.chal[(size_t)k * A.chal_pitch + i];
    uint32_t u = A.u[i];
    GT e1, e2;
    uint32_t res = verify_one<ALGO>(px, py, infbits, ev, ch, u, K, sT, e1, e2, fp32 ? &KF : nullptr);
    A.result[i] = (uint8_t)res;
    if (A.gt) {
      A.gt[i] = (uint8_t)e1.a; A.gt[A.gt_pitch + i] = (uint8_t)e1.b;
      A.gt[2 * A.gt_pitch + i] = (uint8_t)e2.a; A.gt[3 * A.gt_pitch + i] = (uint8_t)e2.b;
    }
  }
}

// Fiat-Shamir verifier: the Challange and rand[0] are replayed from the proof bytes (verify_one_fs)
struct VerifyFsArgs {
  VerifyArgs base;                       // chal, u, bitmap unused
  uint8_t* chal_out; size_t chal_pitch;  // nullable: 6 planes alpha beta gamma z v u (zero for PBH_VR_BAD_ENCODING)
};
// 32 verdict bits of the items w0 .. w0 + 31 (ballot word, little endian) into bitmap bytes w0 / 8 ..; only the bytes of items < n
__device__ __forceinline__ void store_bitmap_word(uint8_t* dst, uint32_t bits, size_t w0, size_t n) {
  if (w0 + 32 <= n) {
    *reinterpret_cast<uint32_t*>(dst) = bits;
  } else {
    for (size_t b = 0; b < (n - w0 + 7) / 8; b++) dst[b] = (uint8_t)(bits >> (8 * b));
  }
}
// BITMAP: the instantiation that also packs the verdict bits into F.base.bitmap (4-byte aligned) and stores every word at the same
// offset of each peer's window.  Its grid-stride loop is warp-uniform so that every iteration ballots 32 consecutive items.  A
// compile-time flag: the plain instantiations compile as they did (see verify_tma_kernel's PEERS).
template <int ALGO, bool BITMAP = false>
__global__ void __launch_bounds__(256, 2) verify_fs_kernel(const Consts K, const ConstsF KF, const bool fp32, const FsSeed seed,
                                                            const Tables* __restrict__ gT, const VerifyFsArgs F, const PeerWindow PW) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  const VerifyArgs& A = F.base;
  auto verify_item = [&](size_t i) -> uint32_t {
    uint32_t px[9], py[9], ev[7];
#pragma unroll
    for (int k = 0; k < 9; k++) {
      px[k] = A.proof[(size_t)(2 * k) * A.proof_pitch + i];
      py[k] = A.proof[(size_t)(2 * k + 1) * A.proof_pitch + i];
    }
    uint32_t infbits = (uint32_t)A.proof[(size_t)18 * A.proof_pitch + i] | ((uint32_t)A.proof[(size_t)19 * A.proof_pitch + i] << 8);
#pragma unroll
    for (int k = 0; k < 7; k++) ev[k] = A.proof[(size_t)(20 + k) * A.proof_pitch + i];
    GT e1, e2;
    uint32_t derived[6];
    uint32_t res = verify_one_fs<ALGO>(px, py, infbits, ev, seed.w, K, sT, e1, e2, fp32 ? &KF : nullptr, derived);
    A.result[i] = (uint8_t)res;
    if (A.gt) {
      A.gt[i] = (uint8_t)e1.a; A.gt[A.gt_pitch + i] = (uint8_t)e1.b;
      A.gt[2 * A.gt_pitch + i] = (uint8_t)e2.a; A.gt[3 * A.gt_pitch + i] = (uint8_t)e2.b;
    }
    if (F.chal_out) {
#pragma unroll
      for (int k = 0; k < 6; k++) F.chal_out[(size_t)k * F.chal_pitch + i] = (uint8_t)derived[k];
    }
    return res;
  };
  if constexpr (!BITMAP) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (size_t)gridDim.x * blockDim.x) verify_item(i);
  } else {
    const int lane = threadIdx.x & 31;
    for (size_t base = (size_t)blockIdx.x * blockDim.x; base < A.n; base += (size_t)gridDim.x * blockDim.x) {
      const size_t i = base + threadIdx.x;
      const bool active = i < A.n;
      const uint32_t res = active ? verify_item(i) : 0u;
      const uint32_t bits = __ballot_sync(0xFFFFFFFFu, active && (res & 1u));
      const size_t w0 = i - lane;                   // first item of this warp: a multiple of 32
      if (lane == 0 && w0 < A.n) {
        store_bitmap_word(A.bitmap + w0 / 8, bits, w0, A.n);
#pragma unroll
        for (uint32_t p = 0; p < 7; p++)            // fixed trip count: delta[] stays in the parameter bank
          if (p < PW.n) store_bitmap_word(A.bitmap + w0 / 8 + PW.delta[p], bits, w0, A.n);
      }
    }
  }
}

// ---- Fiat-Shamir over packed records (include/pbh_b200.h): the codec of pbh_packed.cuh runs in registers around the same per-item
// routines, so no plane ever reaches memory.  12 bytes in and 12 (+4) out per proof, 12 in and 1 out per verification; records are
// read and written as three 32-bit words per thread (a warp touches 384 contiguous bytes), the kernels stay ALU-bound.
template <int ALGO, bool FP32, bool PBH_CIRCUIT>
__global__ void __launch_bounds__(256, 2) prove_fs_packed_kernel(const Consts K, const ConstsF KF, const FsSeed seed, const Tables* __restrict__ gT,
                                                                  size_t n, const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                                  uint32_t* __restrict__ chal_u_out) {
  __shared__ Tables sT;
  __shared__ PackedTables sP;
  stage_packed_tables(&sP);
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint8_t v[21];
    digits17<7>(in[3 * i], v);
    digits17<7>(in[3 * i + 1], v + 7);
    digits17<7>(in[3 * i + 2], v + 14);
    uint32_t w[12], r[9];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 12; k++) { w[k] = v[k]; bad = bad || w[k] >= 17u; }
#pragma unroll
    for (int k = 0; k < 9; k++) { r[k] = v[12 + k]; bad = bad || r[k] >= 17u; }
    if (bad) {
#pragma unroll
      for (int k = 0; k < 12; k++) w[k] = 0;
#pragma unroll
      for (int k = 0; k < 9; k++) r[k] = 0;
    }
    ProofRegs P;
    uint32_t derived[6];
    uint32_t status = prove_item_fs<ALGO, FP32, PBH_CIRCUIT>(w, r, seed.w, K, KF, sT, P, derived, chal_u_out != nullptr);
    if (bad) status = PBH_ST_BAD_ENCODING;
    // the 27 bytes store_proof would write
    const bool ok = status == 0u;
    uint8_t p[27];
    uint32_t inf_lo = 0, inf_hi = 0;
#pragma unroll
    for (int k = 0; k < 9; k++) {
      const uint32_t pw = ok ? P.pt[k] : 0u;
      p[2 * k] = (uint8_t)(pw & 0xFF);
      p[2 * k + 1] = (uint8_t)((pw >> 8) & 0xFF);
      const uint32_t inf = (pw >> 16) & 1u;
      if (k < 8) inf_lo |= inf << k; else inf_hi |= inf;
    }
    p[PBH_PROOF_INF_PLANE] = (uint8_t)inf_lo;
    p[PBH_PROOF_INF_PLANE + 1] = (uint8_t)inf_hi;
#pragma unroll
    for (int k = 0; k < 7; k++) p[PBH_PROOF_EVAL_PLANE + k] = (uint8_t)(ok ? P.ev[k] : 0u);
    uint32_t o[3];
    pack_proof_item(sP, p, (uint8_t)status, o);
    out[3 * i] = o[0];
    out[3 * i + 1] = o[1];
    out[3 * i + 2] = o[2];
    if (chal_u_out) {
      // digits alpha beta gamma z v u, least significant first (pack_chal_u); every derived value is < 17
      uint32_t cu = 0;
#pragma unroll
      for (int k = 5; k >= 0; k--) cu = cu * 17u + derived[k];
      chal_u_out[i] = ok ? cu : 0u;
    }
  }
}

// A packed proof whose status code is not 0 decodes to the all-zero proof and goes through verify_one_fs like any other.
template <int ALGO>
__global__ void __launch_bounds__(256, 2) verify_fs_packed_kernel(const Consts K, const ConstsF KF, const bool fp32, const FsSeed seed,
                                                                   const Tables* __restrict__ gT, size_t n, const uint32_t* __restrict__ proofs,
                                                                   uint8_t* __restrict__ result) {
  __shared__ Tables sT;
  __shared__ PackedTables sP;
  stage_packed_tables(&sP);
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t wd[3] = {proofs[3 * i], proofs[3 * i + 1], proofs[3 * i + 2]};
    uint8_t p[27], st;
    unpack_proof_item(sP, wd, p, &st);
    uint32_t px[9], py[9], ev[7];
#pragma unroll
    for (int k = 0; k < 9; k++) { px[k] = p[2 * k]; py[k] = p[2 * k + 1]; }
    const uint32_t infbits = (uint32_t)p[PBH_PROOF_INF_PLANE] | ((uint32_t)p[PBH_PROOF_INF_PLANE + 1] << 8);
#pragma unroll
    for (int k = 0; k < 7; k++) ev[k] = p[PBH_PROOF_EVAL_PLANE + k];
    GT e1, e2;
    uint32_t derived[6];
    result[i] = (uint8_t)verify_one_fs<ALGO>(px, py, infbits, ev, seed.w, K, sT, e1, e2, fp32 ? &KF : nullptr, derived);
  }
}

// ---- TMA-staged verifier: same tile pipeline as the prover; 33 input planes per item, one result byte out ---------------
struct VerifyTmaMaps {
  CUtensorMap proof, chal, u;
};
struct VerifyTmaSmem {
  alignas(128) uint8_t in[2][34][kTile];    // planes 0..26 proof, 27..31 challenges, 32 u (33 unused: keeps stages 128-byte aligned)
  alignas(8) uint64_t full[2];
  uint32_t tile_of_stage[2];
  alignas(32) uint32_t ballot[2][8];        // the tile's eight verdict words, kept for the peer-window stores
  Tables T;
};
// PEERS: the instantiation that also stores every tile's bitmap bytes into the peers' windows.  A separate instantiation, not
// a run-time branch: the branch alone made the plain verifier 6 % slower at 2^24 items (measured; the compiler emits the tile
// loop twice and schedules both copies worse).
template <int ALGO, int MIN_BLOCKS, bool PEERS>
__global__ void __launch_bounds__(kTile, MIN_BLOCKS) verify_tma_kernel(const __grid_constant__ VerifyTmaMaps M, const Consts K,
                                                                         const ConstsF KF, const bool fp32,
                                                                         const Tables* __restrict__ gT, const VerifyArgs A,
                                                                         unsigned int* __restrict__ tile_counter, const PeerWindow PW) {
  __shared__ VerifyTmaSmem S;
  const int tid = threadIdx.x;
  const size_t tiles = (A.n + kTile - 1) / kTile;
  auto issue = [&](size_t tile, int stage) {
    tma::mbar_arrive_expect_tx(&S.full[stage], 33 * kTile);
    const int32_t c0 = (int32_t)(tile * kTile);
    tma::load_2d(&S.in[stage][0][0], &M.proof, &S.full[stage], c0, 0);
    tma::load_2d(&S.in[stage][27][0], &M.chal, &S.full[stage], c0, 0);
    tma::load_2d(&S.in[stage][32][0], &M.u, &S.full[stage], c0, 0);
  };
  uint32_t pending = 0, t0 = 0;                               // dynamic tile scheduler, see prove_f32_tma_kernel
  if (tid == 0) {
    t0 = atomicAdd(tile_counter, 1u);
    pending = atomicAdd(tile_counter, 1u);
    tma::mbar_init(&S.full[0], 1);
    tma::mbar_init(&S.full[1], 1);
    tma::fence_mbar_init();
  }
  stage_tables(S.T, gT);
  if (tid == 0) {
    S.tile_of_stage[0] = t0;
    if (t0 < tiles) issue(t0, 0);
  }
  __syncthreads();
  uint32_t phase0 = 0, phase1 = 0;
  for (int stage = 0;; stage ^= 1) {
    const size_t tile = S.tile_of_stage[stage];
    if (tile >= tiles) break;
    if (tid == 0) {
      const uint32_t nt = pending;
      S.tile_of_stage[stage ^ 1] = nt;
      if (nt < tiles) {
        issue(nt, stage ^ 1);
        pending = atomicAdd(tile_counter, 1u);
      }
    }
    if (stage == 0) { tma::mbar_wait(&S.full[0], phase0); phase0 ^= 1; } else { tma::mbar_wait(&S.full[1], phase1); phase1 ^= 1; }
    const uint8_t* in = &S.in[stage][0][tid];
    uint32_t px[9], py[9], ev[7], ch[5];
#pragma unroll
    for (int k = 0; k < 9; k++) { px[k] = in[(2 * k) * kTile]; py[k] = in[(2 * k + 1) * kTile]; }
    uint32_t infbits = (uint32_t)in[18 * kTile] | ((uint32_t)in[19 * kTile] << 8);
#pragma unroll
    for (int k = 0; k < 7; k++) ev[k] = in[(20 + k) * kTile];
#pragma unroll
    for (int k = 0; k < 5; k++) ch[k] = in[(27 + k) * kTile];
    uint32_t u = in[32 * kTile];
    GT e1, e2;
    uint32_t res = verify_one<ALGO>(px, py, infbits, ev, ch, u, K, S.T, e1, e2, fp32 ? &KF : nullptr);
    const size_t i = tile * kTile + tid;
    if (i < A.n) {
      A.result[i] = (uint8_t)res;
      if (A.gt) {
        A.gt[i] = (uint8_t)e1.a; A.gt[A.gt_pitch + i] = (uint8_t)e1.b;
        A.gt[2 * A.gt_pitch + i] = (uint8_t)e2.a; A.gt[3 * A.gt_pitch + i] = (uint8_t)e2.b;
      }
    }
    if (A.bitmap != nullptr) {
      // 32 consecutive items per warp: the ballot word is four bitmap bytes (little endian)
      const uint32_t bits = __ballot_sync(0xFFFFFFFFu, i < A.n && (res & 1u));
      const size_t w0 = i - (tid & 31);             // first item of this warp
      if ((tid & 31) == 0 && w0 < A.n) {
        if (w0 + 32 <= A.n) {
          *reinterpret_cast<uint32_t*>(A.bitmap + w0 / 8) = bits;
        } else {
          for (size_t b = 0; b < (A.n - w0 + 7) / 8; b++) A.bitmap[w0 / 8 + b] = (uint8_t)(bits >> (8 * b));
        }
      }
      if (PEERS && (tid & 31) == 0) S.ballot[stage][tid >> 5] = bits;
    }
    __syncthreads();   // every thread has read in[stage]; it may be refilled by the prefetch of the iteration after next
    if (PEERS && A.bitmap != nullptr && tid < 8) {
      // the tile's 32 bitmap bytes go to every peer as one 32-byte store of eight lanes (ballot[stage] is rewritten two
      // iterations from now, behind another block barrier); inline, with the deltas read from the parameter bank: as an
      // out-of-line call taking the window by reference the same stores cost 1.5-2 us per step at N = 2 and 8
      const size_t w0 = tile * kTile + (size_t)tid * 32;
      if (w0 < A.n) {
        const uint32_t word = S.ballot[stage][tid];
#pragma unroll
        for (uint32_t p = 0; p < 7; p++) {
          if (p >= PW.n) continue;
          uint8_t* dst = A.bitmap + w0 / 8 + PW.delta[p];
          if (w0 + 32 <= A.n) {
            *reinterpret_cast<uint32_t*>(dst) = word;
          } else {
            for (size_t b = 0; b < (A.n - w0 + 7) / 8; b++) dst[b] = (uint8_t)(word >> (8 * b));
          }
        }
      }
    }
  }
  tile_scheduler_leave(tile_counter);
}

// ---- sweep kernels -------------------------------------------------------------------------------
// The HBM-bound sweeps (NTT-4 / iNTT-4, polynomial add, division by Z_H) work on four items at once: one 32-bit word
// per plane holds the same coefficient of four consecutive items in its byte lanes, and all F_17 arithmetic is byte-lane
// SWAR on the integer ALU pipe.  16 = -1 (mod 17), so a lane value x = 16a + b folds to b - a, the size-4 twiddles
// are +-1 and +-4 (a 2-bit lane shift), and -c is 17 - c.  No multiplies, no cross-lane carries (bounds in comments).

// every byte lane (0..255) -> its residue mod 17 (0..16)
__device__ __forceinline__ uint32_t swar_mod17(uint32_t x) {
  const uint32_t lo = x & 0x0F0F0F0Fu, hi = (x >> 4) & 0x0F0F0F0Fu;
  const uint32_t t = lo + 0x11111111u - hi;                 // b - a + 17, lanes in [2, 32]
  const uint32_t m = (t + 0x6F6F6F6Fu) & 0x80808080u;       // lane >= 17  <=>  lane + 111 >= 128
  return t - ((m >> 7) + (m >> 3));                         // subtract 17 (= 1 + 16) from the flagged lanes
}
__device__ __forceinline__ uint32_t swar_neg17(uint32_t x) { return 0x11111111u - x; }   // lanes 0..16 -> 17 - lane (1..17)

// lanes 0..16 times the constant C (0 < C < 17): lanes congruent to C x, at most 255, by shifts and adds (-c is 17 - c)
template <int C>
__device__ __forceinline__ uint32_t swar_mulc(uint32_t x) {
  static_assert(C >= 1 && C <= 16, "F_17 constant");
  switch (C) {
    case 1: return x;
    case 2: return x << 1;
    case 3: return x + (x << 1);
    case 4: return x << 2;
    case 5: return x + (x << 2);
    case 6: return (x << 1) + (x << 2);
    case 7: return (x << 3) + swar_neg17(x);                 // 8x - x = 8x + (17 - x), lanes <= 145
    case 8: return x << 3;
    case 9: return x + (x << 3);
    case 10: return (x << 1) + (x << 3);
    case 11: return swar_mulc<6>(swar_neg17(x));              // -6 (17 - x <= 17: lanes <= 102)
    case 12: return (x << 2) + (x << 3);
    case 13: return swar_neg17(x) << 2;                       // -4
    case 14: return swar_mulc<3>(swar_neg17(x));              // -3
    case 15: return swar_neg17(x) << 1;                       // -2
    default: return swar_neg17(x);                            // -1
  }
}
// lanes 0..255 -> lanes congruent to -4 x (= x / 4: 13 = 1/4 = -4), in 8..128, WITHOUT reducing x first: x = 16 a + b = b - a,
// so -4 x = 4 a + 4 (17 - b); one lane reduction fewer per output of the inverse transform
__device__ __forceinline__ uint32_t swar_m4(uint32_t x) {
  const uint32_t lo = x & 0x0F0F0F0Fu, hi = (x >> 4) & 0x0F0F0F0Fu;
  return ((hi + 0x11111111u) - lo) << 2;                      // lanes (a + 17 - b) <= 32, times 4 <= 128: no carry between lanes
}
__host__ __device__ constexpr int pow17(int b, int e) { int r = 1; for (int i = 0; i < e; i++) r = r * b % 17; return r; }
__host__ __device__ constexpr int inv17c_(int a) { return pow17(a, 15); }

// Size-4 transforms over F_17 with omega = 4 on the coset K H, K in {1, 2, 3}: K = 1 is H itself (src/fft.rs:66-106 with
// EvaluationDomainGenerator(4, 4); the inverse is Plonk::interpolate_at_h, src/plonk.rs:177-179), K = 2 and K = 3 are the
// cosets k1 H = {2, 8, 15, 9} and k2 H = {3, 12, 14, 5} of src/plonk.rs:136-139 (K1, K2 of src/pbh/mod.rs:27-28).
//   forward: e_i = p(K 4^i) = sum_j (c_j K^j) 4^(ij)         - the plain transform of the coefficients scaled by K^j
//   inverse: c_j = K^-j * 13 sum_i 4^(-ij) v_i, 13 = 1/4     - the plain inverse, its 1/4 folded with K^-j into ONE constant
// so the inverse costs the same as on H, and the forward transform costs three more lane reductions.
template <bool INVERSE, int K>
__device__ __forceinline__ void swar_ntt4(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t (&o)[4]) {
  w0 = swar_mod17(w0); w1 = swar_mod17(w1); w2 = swar_mod17(w2); w3 = swar_mod17(w3);   // any byte value is accepted
  if (!INVERSE && K != 1) {
    w1 = swar_mod17(swar_mulc<pow17(K, 1)>(w1)); w2 = swar_mod17(swar_mulc<pow17(K, 2)>(w2)); w3 = swar_mod17(swar_mulc<pow17(K, 3)>(w3));
  }
  const uint32_t n1 = swar_neg17(w1), n2 = swar_neg17(w2), n3 = swar_neg17(w3);
  const uint32_t s0 = w0 + w1 + w2 + w3;                            // lanes <= 64
  const uint32_t sp = w0 + (w1 << 2) + n2 + (n3 << 2);              // c0 + 4c1 - c2 - 4c3, lanes <= 165
  const uint32_t s2 = w0 + n1 + w2 + n3;                            // c0 - c1 + c2 - c3,   lanes <= 66
  const uint32_t sm = w0 + (n1 << 2) + n2 + (w3 << 2);              // c0 - 4c1 - c2 + 4c3, lanes <= 165
  if (!INVERSE) {
    o[0] = swar_mod17(s0); o[1] = swar_mod17(sp); o[2] = swar_mod17(s2); o[3] = swar_mod17(sm);
  } else {
    // omega^-1 = -4 swaps the roles of sp and sm; then one constant per coefficient: 13 K^-j
    o[0] = swar_mod17(swar_m4(s0));
    if (K == 1) {
      o[1] = swar_mod17(swar_m4(sm)); o[2] = swar_mod17(swar_m4(s2)); o[3] = swar_mod17(swar_m4(sp));
    } else {
      o[1] = swar_mod17(swar_mulc<13 * inv17c_(pow17(K, 1)) % 17>(swar_mod17(sm)));
      o[2] = swar_mod17(swar_mulc<13 * inv17c_(pow17(K, 2)) % 17>(swar_mod17(s2)));
      o[3] = swar_mod17(swar_mulc<13 * inv17c_(pow17(K, 3)) % 17>(swar_mod17(sp)));
    }
  }
}

// vec: 0 = byte path, 4 = one 32-bit word per plane and thread (4 items), 16 = one 128-bit word (16 items; needs
// 16-byte aligned bases and pitches).  Wider accesses keep more bytes in flight per thread: the kernel is
// latency-limited, not ALU-limited.
template <bool INVERSE, int K>
__global__ void __launch_bounds__(kBlock) ntt4_kernel(size_t n, const uint8_t* __restrict__ in, size_t in_pitch,
                                                       uint8_t* __restrict__ out, size_t out_pitch, int vec) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t done = 0;
  if (vec == 16) {
    const size_t n16 = n / 16;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n16; q += stride) {
      uint4 wv[4], ov[4];
#pragma unroll
      for (int k = 0; k < 4; k++) wv[k] = reinterpret_cast<const uint4*>(in + (size_t)k * in_pitch)[q];
      uint32_t o[4];
      swar_ntt4<INVERSE, K>(wv[0].x, wv[1].x, wv[2].x, wv[3].x, o); ov[0].x = o[0]; ov[1].x = o[1]; ov[2].x = o[2]; ov[3].x = o[3];
      swar_ntt4<INVERSE, K>(wv[0].y, wv[1].y, wv[2].y, wv[3].y, o); ov[0].y = o[0]; ov[1].y = o[1]; ov[2].y = o[2]; ov[3].y = o[3];
      swar_ntt4<INVERSE, K>(wv[0].z, wv[1].z, wv[2].z, wv[3].z, o); ov[0].z = o[0]; ov[1].z = o[1]; ov[2].z = o[2]; ov[3].z = o[3];
      swar_ntt4<INVERSE, K>(wv[0].w, wv[1].w, wv[2].w, wv[3].w, o); ov[0].w = o[0]; ov[1].w = o[1]; ov[2].w = o[2]; ov[3].w = o[3];
#pragma unroll
      for (int k = 0; k < 4; k++) reinterpret_cast<uint4*>(out + (size_t)k * out_pitch)[q] = ov[k];
    }
    done = n16 * 16;
  } else if (vec == 4) {
    const size_t n4 = n / 4;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += stride) {
      uint32_t wv[4], ov[4];
#pragma unroll
      for (int k = 0; k < 4; k++) wv[k] = reinterpret_cast<const uint32_t*>(in + (size_t)k * in_pitch)[q];
      swar_ntt4<INVERSE, K>(wv[0], wv[1], wv[2], wv[3], ov);
#pragma unroll
      for (int k = 0; k < 4; k++) reinterpret_cast<uint32_t*>(out + (size_t)k * out_pitch)[q] = ov[k];
    }
    done = n4 * 4;
  }
  for (size_t i = done + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    uint32_t ov[4];
    swar_ntt4<INVERSE, K>(in[i], in[in_pitch + i], in[2 * in_pitch + i], in[3 * in_pitch + i], ov);   // one live lane
#pragma unroll
    for (int k = 0; k < 4; k++) out[(size_t)k * out_pitch + i] = (uint8_t)ov[k];
  }
}

// generic power-of-two NTT over F_m (m < 2^16), size <= 64, one item per thread, values in local memory
// (src/fft.rs:66-78, 90-106: radix-2 decimation in time, then for the inverse reverse-and-scale).
__global__ void __launch_bounds__(kBlock) ntt_generic_kernel(size_t n, uint32_t modulus, uint32_t size, uint32_t log2size,
                                                              uint32_t len_inv, int inverse, const uint16_t* __restrict__ tw,
                                                              const uint16_t* __restrict__ in, size_t in_pitch,
                                                              uint16_t* __restrict__ out, size_t out_pitch) {
  __shared__ uint32_t s_tw[64];
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_tw[i] = i < (int)size ? tw[i] : 0;
  __syncthreads();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t a[64];
    // bit-reversed load = the even/odd splits of the recursion
    for (uint32_t k = 0; k < size; k++) {
      uint32_t r = __brev(k) >> (32 - log2size);
      a[r] = in[(size_t)k * in_pitch + i] % modulus;
    }
    for (uint32_t len = 2; len <= size; len <<= 1) {
      uint32_t step = size / len;   // domain of this level is every step-th power
      for (uint32_t base = 0; base < size; base += len) {
        for (uint32_t j = 0; j < len / 2; j++) {
          uint32_t x = a[base + j];
          uint32_t y = (uint32_t)(((uint64_t)a[base + j + len / 2] * s_tw[j * step]) % modulus);
          a[base + j] = (x + y) % modulus;
          a[base + j + len / 2] = (x + modulus - y) % modulus;
        }
      }
    }
    if (inverse) {
      // vals[0], then vals reversed, each times len^-1                       src/fft.rs:72-78
      for (uint32_t k = 0; k < size; k++) {
        uint32_t src = k == 0 ? 0 : size - k;
        out[(size_t)k * out_pitch + i] = (uint16_t)(((uint64_t)a[src] * len_inv) % modulus);
      }
    } else {
      for (uint32_t k = 0; k < size; k++) out[(size_t)k * out_pitch + i] = (uint16_t)a[k];
    }
  }
}

// mul_ntt (src/fft.rs:109-132) over CooleyTurkey: both operands zero-extended to `size` = la + lb values, transformed,
// multiplied pointwise and transformed back (fft_inv = forward transform, reverse, scale: src/fft.rs:72-78).
__device__ __forceinline__ void ntt_dit_inplace(uint32_t (&a)[64], uint32_t size, uint32_t modulus, const uint32_t* s_tw) {
  for (uint32_t len = 2; len <= size; len <<= 1) {
    uint32_t step = size / len;
    for (uint32_t base = 0; base < size; base += len) {
      for (uint32_t j = 0; j < len / 2; j++) {
        uint32_t x = a[base + j];
        uint32_t y = (uint32_t)(((uint64_t)a[base + j + len / 2] * s_tw[j * step]) % modulus);
        a[base + j] = (x + y) % modulus;
        a[base + j + len / 2] = (x + modulus - y) % modulus;
      }
    }
  }
}
__global__ void __launch_bounds__(kBlock) mul_ntt_kernel(size_t n, uint32_t modulus, uint32_t size, uint32_t log2size, uint32_t len_inv,
                                                          uint32_t la, uint32_t lb, const uint16_t* __restrict__ tw,
                                                          const uint16_t* __restrict__ a_in, size_t a_pitch,
                                                          const uint16_t* __restrict__ b_in, size_t b_pitch, uint16_t* __restrict__ out,
                                                          size_t out_pitch) {
  __shared__ uint32_t s_tw[64];
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_tw[i] = i < (int)size ? tw[i] : 0;
  __syncthreads();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t a[64], b[64];
    for (uint32_t k = 0; k < size; k++) {
      uint32_t r = __brev(k) >> (32 - log2size);
      a[r] = k < la ? a_in[(size_t)k * a_pitch + i] % modulus : 0u;
      b[r] = k < lb ? b_in[(size_t)k * b_pitch + i] % modulus : 0u;
    }
    ntt_dit_inplace(a, size, modulus, s_tw);
    ntt_dit_inplace(b, size, modulus, s_tw);
    for (uint32_t k = 0; k < size; k++) {           // pointwise product, stored bit-reversed for the second transform
      uint32_t r = __brev(k) >> (32 - log2size);
      if (r >= k) {
        uint32_t ck = (uint32_t)(((uint64_t)a[k] * b[k]) % modulus), cr = (uint32_t)(((uint64_t)a[r] * b[r]) % modulus);
        a[k] = cr; a[r] = ck;
      }
    }
    ntt_dit_inplace(a, size, modulus, s_tw);
    for (uint32_t k = 0; k < size; k++) {
      uint32_t src = k == 0 ? 0 : size - k;
      out[(size_t)k * out_pitch + i] = (uint16_t)(((uint64_t)a[src] * len_inv) % modulus);
    }
  }
}

// Poly * scalar (src/poly.rs:220-228), Poly::eval (src/poly.rs:71-79) and Poly / (x - c) (src/poly.rs:230-247 with the
// monic linear divisors of src/plonk.rs:437-442) over F_17: `len` coefficient planes followed by one operand plane
// (the scalar, the point, c), four items per 32-bit word.  OP 0: len planes out; OP 1: one plane out; OP 2: len - 1
// quotient planes then the remainder plane (a Horner chain whose intermediate values are the quotient).
//
// Arithmetic: every item has its OWN multiplier, which rules out byte-lane SWAR multiplies, and one int32 multiply +
// reduction per byte made round 1's version ALU-bound at 94-175 instructions per item (profiles/r02a_sweeps_before.txt).
// Here two items share one packed-half instruction: a byte b becomes the half 1024 + b by planting the exponent byte 0x64
// next to it (one PRMT for two lanes), all values are integers below 2048 in magnitude and therefore exact in fp16, and
// x mod 17 is three HFMA2-class instructions for two lanes (round(x / 17) with the 1536 = 1.5 * 2^10 rounding constant,
// exact for |x| <= 2048: checked for every integer of the range by the CPU test suite).  Any input byte is
// accepted: |acc * x + c| <= 8 * 8 + 255 and |c * x| <= 255 * 8.
__device__ __forceinline__ __half2 h2_bits(uint32_t b) { return *reinterpret_cast<__half2*>(&b); }
__device__ __forceinline__ uint32_t h2_word(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
// bytes (0, 1) or (2, 3) of w as two exact halves
__device__ __forceinline__ __half2 h2_from_bytes(uint32_t w, bool upper) {
  return __hsub2(h2_bits(__byte_perm(w, 0x64646464u, upper ? 0x4342u : 0x4140u)), h2_bits(0x64006400u));
}
// centred residue mod 17 of two exact integers |x| <= 2048
__device__ __forceinline__ __half2 h2_red17(__half2 x) {
  const __half2 k = h2_bits(0x66006600u);                                 // 1536, 1536
  const __half2 q = __hsub2(__hfma2(x, h2_bits(0x2B882B88u), k), k);      // 0x2B88 = fp16(1 / 17) = 0.05883789
  return __hfma2(q, h2_bits(0xCC40CC40u), x);                             // 0xCC40 = -17
}
// four centred residues -> canonical bytes 0..16 packed in one word
__device__ __forceinline__ uint32_t h2_pack_canon(__half2 a01, __half2 a23) {
  const __half2 zero = h2_bits(0u), p17 = h2_bits(0x4C404C40u), bias = h2_bits(0x64006400u);
  a01 = __hadd2(__hfma2(__hlt2(a01, zero), p17, a01), bias);
  a23 = __hadd2(__hfma2(__hlt2(a23, zero), p17, a23), bias);
  return __byte_perm(h2_word(a01), h2_word(a23), 0x6420u);
}
// WORDS 32-bit words per plane and thread: 1 (4 items, 4-byte aligned planes) or 4 (16 items through one 128-bit access,
// 16-byte aligned planes: four times the bytes in flight per thread and a quarter of the address arithmetic per item).
template <int WORDS> struct PlaneVec;
template <> struct PlaneVec<1> {
  uint32_t w[1];
  __device__ __forceinline__ void load(const uint8_t* p, size_t q) { w[0] = reinterpret_cast<const uint32_t*>(p)[q]; }
  __device__ __forceinline__ void store(uint8_t* p, size_t q) const { reinterpret_cast<uint32_t*>(p)[q] = w[0]; }
};
template <> struct PlaneVec<4> {
  uint32_t w[4];
  __device__ __forceinline__ void load(const uint8_t* p, size_t q) { const uint4 v = reinterpret_cast<const uint4*>(p)[q]; w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
  __device__ __forceinline__ void store(uint8_t* p, size_t q) const { reinterpret_cast<uint4*>(p)[q] = make_uint4(w[0], w[1], w[2], w[3]); }
};
template <int OP, int WORDS>
__device__ __forceinline__ void poly_unary_vec(size_t q, uint32_t len, const uint8_t* __restrict__ in, size_t in_pitch, uint8_t* __restrict__ out,
                                               size_t out_pitch) {
  PlaneVec<WORDS> op;
  op.load(in + (size_t)len * in_pitch, q);
  __half2 x[2 * WORDS], acc[2 * WORDS];
#pragma unroll
  for (int j = 0; j < WORDS; j++) {
    x[2 * j] = h2_red17(h2_from_bytes(op.w[j], false)); x[2 * j + 1] = h2_red17(h2_from_bytes(op.w[j], true));
    acc[2 * j] = acc[2 * j + 1] = h2_bits(0u);
  }
  constexpr uint32_t kAhead = WORDS == 1 ? 8 : 4;     // planes whose loads are issued before any is consumed
  if (OP == 0) {
    for (uint32_t k0 = 0; k0 < len; k0 += kAhead) {
      PlaneVec<WORDS> v[kAhead];
#pragma unroll
      for (uint32_t j = 0; j < kAhead; j++)
        if (k0 + j < len) v[j].load(in + (size_t)(k0 + j) * in_pitch, q);
#pragma unroll
      for (uint32_t j = 0; j < kAhead; j++) {
        if (k0 + j < len) {
          PlaneVec<WORDS> o;
#pragma unroll
          for (int t = 0; t < WORDS; t++)
            o.w[t] = h2_pack_canon(h2_red17(__hmul2(h2_from_bytes(v[j].w[t], false), x[2 * t])), h2_red17(__hmul2(h2_from_bytes(v[j].w[t], true), x[2 * t + 1])));
          o.store(out + (size_t)(k0 + j) * out_pitch, q);
        }
      }
    }
  } else {
    for (uint32_t k0 = len; k0 > 0; k0 = k0 > kAhead ? k0 - kAhead : 0) {   // planes k0-1, k0-2, ... (Horner runs downwards)
      PlaneVec<WORDS> v[kAhead];
#pragma unroll
      for (uint32_t j = 0; j < kAhead; j++)
        if (j < k0) v[j].load(in + (size_t)(k0 - 1 - j) * in_pitch, q);
#pragma unroll
      for (uint32_t j = 0; j < kAhead; j++) {
        if (j < k0) {
          const uint32_t k = k0 - 1 - j;
          if (OP == 2 && k + 1 < len) {
            PlaneVec<WORDS> o;
#pragma unroll
            for (int t = 0; t < WORDS; t++) o.w[t] = h2_pack_canon(acc[2 * t], acc[2 * t + 1]);
            o.store(out + (size_t)k * out_pitch, q);
          }
#pragma unroll
          for (int t = 0; t < WORDS; t++) {
            acc[2 * t] = h2_red17(__hfma2(acc[2 * t], x[2 * t], h2_from_bytes(v[j].w[t], false)));
            acc[2 * t + 1] = h2_red17(__hfma2(acc[2 * t + 1], x[2 * t + 1], h2_from_bytes(v[j].w[t], true)));
          }
        }
      }
    }
    PlaneVec<WORDS> o;
#pragma unroll
    for (int t = 0; t < WORDS; t++) o.w[t] = h2_pack_canon(acc[2 * t], acc[2 * t + 1]);
    o.store(out + (size_t)(OP == 2 ? len - 1 : 0) * out_pitch, q);
  }
}
// vec: 0 = byte path only, 4 = one 32-bit word per plane and thread, 16 = one 128-bit word
template <int OP>
__global__ void __launch_bounds__(kBlock) poly_unary_kernel(size_t n, uint32_t len, const uint8_t* __restrict__ in, size_t in_pitch,
                                                             uint8_t* __restrict__ out, size_t out_pitch, int vec) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t done = 0;
  if (vec == 16) {
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n / 16; q += stride) poly_unary_vec<OP, 4>(q, len, in, in_pitch, out, out_pitch);
    done = n / 16 * 16;
  } else if (vec == 4) {
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n / 4; q += stride) poly_unary_vec<OP, 1>(q, len, in, in_pitch, out, out_pitch);
    done = n / 4 * 4;
  }
  for (size_t i = done + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t x = mod17(in[(size_t)len * in_pitch + i]);
    if (OP == 0) {
      for (uint32_t k = 0; k < len; k++) out[(size_t)k * out_pitch + i] = (uint8_t)mod17(mod17(in[(size_t)k * in_pitch + i]) * x);
    } else {
      uint32_t acc = 0;
      for (uint32_t k = len; k-- > 0;) {
        if (OP == 2 && k + 1 < len) out[(size_t)k * out_pitch + i] = (uint8_t)acc;
        acc = mod17(acc * x + mod17(in[(size_t)k * in_pitch + i]));
      }
      out[(size_t)(OP == 2 ? len - 1 : 0) * out_pitch + i] = (uint8_t)acc;
    }
  }
}

// schoolbook product over F_17, runtime lengths <= 16                        src/poly.rs:205-218
__global__ void __launch_bounds__(kBlock) poly_mul_kernel(size_t n, uint32_t la, uint32_t lb, const uint8_t* __restrict__ a,
                                                           size_t a_pitch, const uint8_t* __restrict__ b, size_t b_pitch,
                                                           uint8_t* __restrict__ out, size_t out_pitch) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t av[16], bv[16];
#pragma unroll
    for (uint32_t k = 0; k < 16; k++) {
      av[k] = k < la ? a[(size_t)k * a_pitch + i] : 0u;
      bv[k] = k < lb ? b[(size_t)k * b_pitch + i] : 0u;
    }
#pragma unroll
    for (uint32_t k = 0; k < 31; k++) {
      if (k < la + lb - 1) {
        uint32_t acc = 0;
#pragma unroll
        for (uint32_t j = 0; j < 16; j++) {
          if (j <= k && k - j < 16) acc += av[j] * bv[k - j];
        }
        out[(size_t)k * out_pitch + i] = (uint8_t)mod17(acc);
      }
    }
  }
}

// The same product for LA, LB <= 8 (padded to even sizes by the host), four items per 32-bit word and exact FP32
// arithmetic: round 1's kernel above keeps its operand lengths in registers and executed 560 instructions per 6 x 6 product
// (profiles/r02a_sweeps_before.txt).  Input bytes are used as they are (any value: 8 x 255^2 < 2^20), every output is
// reduced once with a FLOOR reduction that lands on the canonical residue 0..16 directly (the operands are non-negative:
// q = rint((x - 8) / 17) is floor(x / 17) because the fractional parts of x / 17 are multiples of 1 / 17), and the four
// lanes of an output word are packed by planting them under the 2^23 exponent.
__device__ __forceinline__ float f_byte(uint32_t w, int k) { return __int_as_float((int)__byte_perm(w, 0x4B000000u, 0x7440u + (uint32_t)k)) - 8388608.0f; }
__device__ __forceinline__ uint32_t f_floor_mod17_biased(float xm8) {    // xm8 = x - 8 for an exact integer 0 <= x < 2^20: bits of 2^23 + (x mod 17)
  const float q = fmaf(xm8, 0.058823529411764705f, 12582912.0f) - 12582912.0f;    // rint((x - 8) / 17) = floor(x / 17)
  return (uint32_t)__float_as_int(fmaf(q, -17.0f, xm8) + 8388616.0f);             // x - 8 - 17 q + 8 + 2^23
}
template <int LA, int LB>
__global__ void __launch_bounds__(kBlock) poly_mul_vec_kernel(size_t n4, uint32_t la, uint32_t lb, const uint8_t* __restrict__ a, size_t a_pitch,
                                                               const uint8_t* __restrict__ b, size_t b_pitch, uint8_t* __restrict__ out,
                                                               size_t out_pitch) {
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += (size_t)gridDim.x * blockDim.x) {
    uint32_t aw[LA], bw[LB];
#pragma unroll
    for (int k = 0; k < LA; k++) aw[k] = (uint32_t)k < la ? reinterpret_cast<const uint32_t*>(a + (size_t)k * a_pitch)[q] : 0u;
#pragma unroll
    for (int k = 0; k < LB; k++) bw[k] = (uint32_t)k < lb ? reinterpret_cast<const uint32_t*>(b + (size_t)k * b_pitch)[q] : 0u;
    float av[4][LA], bv[4][LB];
#pragma unroll
    for (int l = 0; l < 4; l++) {
#pragma unroll
      for (int k = 0; k < LA; k++) av[l][k] = f_byte(aw[k], l);
#pragma unroll
      for (int k = 0; k < LB; k++) bv[l][k] = f_byte(bw[k], l);
    }
#pragma unroll
    for (int k = 0; k < LA + LB - 1; k++) {
      if ((uint32_t)k < la + lb - 1) {
        uint32_t r[4];
#pragma unroll
        for (int l = 0; l < 4; l++) {
          float acc = -8.0f;                                   // the floor reduction takes x - 8
#pragma unroll
          for (int i = 0; i < LA; i++)
            if (k - i >= 0 && k - i < LB) acc = fmaf(av[l][i], bv[l][k - i], acc);
          r[l] = f_floor_mod17_biased(acc);
        }
        reinterpret_cast<uint32_t*>(out + (size_t)k * out_pitch)[q] = __byte_perm(__byte_perm(r[0], r[1], 0x0040u), __byte_perm(r[2], r[3], 0x0040u), 0x5410u);
      }
    }
  }
}

// coefficientwise a + b or a - b on `len` planes, four items per word                     src/poly.rs:165-203
__global__ void __launch_bounds__(kBlock) poly_add_kernel(size_t n, uint32_t len, int subtract, const uint8_t* __restrict__ a,
                                                           size_t a_pitch, const uint8_t* __restrict__ b, size_t b_pitch,
                                                           uint8_t* __restrict__ out, size_t out_pitch, bool vec_ok) {
  const size_t n4 = vec_ok ? n / 4 : 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += stride) {
    for (uint32_t k0 = 0; k0 < len; k0 += 8) {      // eight planes' loads are issued before any is consumed
      uint32_t x[8], y[8];
#pragma unroll
      for (uint32_t j = 0; j < 8; j++) {
        const bool live = k0 + j < len;
        x[j] = live ? reinterpret_cast<const uint32_t*>(a + (size_t)(k0 + j) * a_pitch)[q] : 0u;
        y[j] = live ? reinterpret_cast<const uint32_t*>(b + (size_t)(k0 + j) * b_pitch)[q] : 0u;
      }
#pragma unroll
      for (uint32_t j = 0; j < 8; j++) {
        if (k0 + j < len) {
          const uint32_t yy = swar_mod17(y[j]);
          reinterpret_cast<uint32_t*>(out + (size_t)(k0 + j) * out_pitch)[q] = swar_mod17(swar_mod17(x[j]) + (subtract ? swar_neg17(yy) : yy));
        }
      }
    }
  }
  for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    for (uint32_t k = 0; k < len; k++) {
      uint32_t x = swar_mod17(a[(size_t)k * a_pitch + i]), y = swar_mod17(b[(size_t)k * b_pitch + i]);
      out[(size_t)k * out_pitch + i] = (uint8_t)swar_mod17(x + (subtract ? swar_neg17(y) : y));
    }
  }
}

// (q, r) = p / (x^4 - 1): 22 planes -> 18 + 4 planes, four items per word          src/poly.rs:230-247, src/plonk.rs:369
template <class W>
__device__ __forceinline__ void swar_div_zh(const W (&num)[22], W (&t)[18], W (&r)[4]) {
  // t[j] = num[j+4] + t[j+4]: at most 5 residues accumulate (lanes <= 80) before the fold
#pragma unroll
  for (int j = 17; j >= 0; j--) t[j] = (j + 4 < 18) ? swar_mod17(num[j + 4] + t[j + 4]) : num[j + 4];
#pragma unroll
  for (int j = 0; j < 4; j++) r[j] = swar_mod17(num[j] + t[j]);
}
__global__ void __launch_bounds__(kBlock) poly_div_zh_kernel(size_t n, const uint8_t* __restrict__ p, size_t p_pitch,
                                                              uint8_t* __restrict__ q, size_t q_pitch, uint8_t* __restrict__ r,
                                                              size_t r_pitch, bool vec_ok) {
  const size_t n4 = vec_ok ? n / 4 : 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < n4; w += stride) {
    uint32_t num[22], t[18], rem[4];
#pragma unroll
    for (int k = 0; k < 22; k++) num[k] = swar_mod17(reinterpret_cast<const uint32_t*>(p + (size_t)k * p_pitch)[w]);
    swar_div_zh(num, t, rem);
#pragma unroll
    for (int j = 0; j < 18; j++) reinterpret_cast<uint32_t*>(q + (size_t)j * q_pitch)[w] = t[j];
#pragma unroll
    for (int j = 0; j < 4; j++) reinterpret_cast<uint32_t*>(r + (size_t)j * r_pitch)[w] = rem[j];
  }
  for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    uint32_t num[22], t[18], rem[4];
#pragma unroll
    for (int k = 0; k < 22; k++) num[k] = swar_mod17(p[(size_t)k * p_pitch + i]);
    swar_div_zh(num, t, rem);
#pragma unroll
    for (int j = 0; j < 18; j++) q[(size_t)j * q_pitch + i] = (uint8_t)t[j];
#pragma unroll
    for (int j = 0; j < 4; j++) r[(size_t)j * r_pitch + i] = (uint8_t)rem[j];
  }
}

// G1P * F101, src/pbh/g1.rs:146-168; scalar 0..100 (7 bits)
__global__ void __launch_bounds__(kBlock) g1_smul_kernel(const Tables* __restrict__ gT, size_t n, const uint8_t* __restrict__ in,
                                                          size_t in_pitch, uint8_t* __restrict__ out, size_t out_pitch) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    // exact FP32 curve arithmetic (pbh_g1f.cuh): every multiple of one point lies on one curve y^2 = x^3 + b', whatever b' is
    // (the addition formulas never use b), so the unified slope serves any (x, y), on the reference's curve or not
    F32* tag = nullptr;
    G1F<F32> p;
    p.x = f_from_u32(in[i] % 101u, tag); p.y = f_from_u32(in[in_pitch + i] % 101u, tag); p.inf = in[2 * in_pitch + i] != 0;
    const uint32_t k = in[3 * in_pitch + i] % 101u;
    const G1F<F32> r = g1f_smul<7>(p, k, sT.inv101c);
    out[i] = (uint8_t)f_canon101(r.x); out[out_pitch + i] = (uint8_t)f_canon101(r.y); out[2 * out_pitch + i] = (uint8_t)(r.inf ? 1 : 0);
  }
}

// G1P + G1P, src/pbh/g1.rs:119-144
__global__ void __launch_bounds__(kBlock) g1_add_kernel(const Tables* __restrict__ gT, size_t n, const uint8_t* __restrict__ in,
                                                         size_t in_pitch, uint8_t* __restrict__ out, size_t out_pitch) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    G1 p, q;
    p.x = in[i] % 101u; p.y = in[in_pitch + i] % 101u; p.inf = in[2 * in_pitch + i] != 0;
    q.x = in[3 * in_pitch + i] % 101u; q.y = in[4 * in_pitch + i] % 101u; q.inf = in[5 * in_pitch + i] != 0;
    bool bad;
    G1 r = g1_add(p, q, sT.inv101, &bad);
    if (bad) { r.x = 0; r.y = 0; r.inf = 0xFF; }
    out[i] = (uint8_t)r.x; out[out_pitch + i] = (uint8_t)r.y; out[2 * out_pitch + i] = (uint8_t)r.inf;
  }
}

// SRS::eval_at_s over 7 coefficient planes, src/plonk.rs:51-58.  inf = 0xFF where the reference indexes out of bounds.
template <int ALGO>
__global__ void __launch_bounds__(kBlock) kzg_commit_kernel(const Consts K, const Tables* __restrict__ gT, size_t n,
                                                             const uint8_t* __restrict__ in, size_t in_pitch,
                                                             uint8_t* __restrict__ out, size_t out_pitch) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t c[7];
#pragma unroll
    for (int k = 0; k < 7; k++) c[k] = mod17(in[(size_t)k * in_pitch + i]);
    uint32_t w = (ALGO == ALGO_TABLE) ? commit<ALGO_TABLE>(c, K, sT) : commit_pairs_f32<7>(c, sT);
    if (longer_than(c, K.n_pts)) w = 0xFF0000u;
    out[i] = (uint8_t)(w & 0xFF); out[out_pitch + i] = (uint8_t)((w >> 8) & 0xFF); out[2 * out_pitch + i] = (uint8_t)(w >> 16);
  }
}

// The same commitment for PBH_ALGO_TABLE with at least 7 SRS points, four items per 32-bit word: the exponent of G is
// the dot product of the coefficients with the SRS discrete logs, accumulated in two 16-bit lanes per word (any byte
// value is accepted: 7 * 255 * 16 < 2^16), reduced with 16 = -1 (mod 17), and the point comes from the 17-entry table.
// One-byte accesses keep too few bytes in flight to cover the HBM latency (measured 2.2 TB/s); words quadruple them.
__global__ void __launch_bounds__(kBlock) kzg_commit_table_vec_kernel(const Consts K, const Tables* __restrict__ gT, size_t n4,
                                                                       const uint8_t* __restrict__ in, size_t in_pitch,
                                                                       uint8_t* __restrict__ out, size_t out_pitch) {
  __shared__ uint32_t s_pt[17];
  if (threadIdx.x < 17) s_pt[threadIdx.x] = gT->pt17[threadIdx.x];
  __syncthreads();
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += (size_t)gridDim.x * blockDim.x) {
    uint32_t w[7];
#pragma unroll
    for (int k = 0; k < 7; k++) w[k] = reinterpret_cast<const uint32_t*>(in + (size_t)k * in_pitch)[q];
    uint32_t ev = 0, od = 0;   // items 0, 2 and items 1, 3 as 16-bit lanes
#pragma unroll
    for (int k = 0; k < 7; k++) {
      ev += (w[k] & 0x00FF00FFu) * K.srs_dlog[k];
      od += ((w[k] >> 8) & 0x00FF00FFu) * K.srs_dlog[k];
    }
    // x = n0 + 16 n1 + 256 n2 + 4096 n3 = n0 - n1 + n2 - n3 (mod 17); + 34 keeps the lane positive (<= 64)
    const uint32_t m = 0x000F000Fu;
    const uint32_t te = (ev & m) + ((ev >> 8) & m) + 0x00220022u - ((ev >> 4) & m) - ((ev >> 12) & m);
    const uint32_t to = (od & m) + ((od >> 8) & m) + 0x00220022u - ((od >> 4) & m) - ((od >> 12) & m);
    const uint32_t e = swar_mod17(te | (to << 8));   // byte lane j = exponent of item j
    const uint32_t p0 = s_pt[e & 0xFFu], p1 = s_pt[(e >> 8) & 0xFFu], p2 = s_pt[(e >> 16) & 0xFFu], p3 = s_pt[e >> 24];
    // transpose the four packed points (x | y << 8 | inf << 16) into the three output planes
    const uint32_t a01 = __byte_perm(p0, p1, 0x5140), a23 = __byte_perm(p2, p3, 0x5140);   // x0 x1 y0 y1 / x2 x3 y2 y3
    reinterpret_cast<uint32_t*>(out)[q] = __byte_perm(a01, a23, 0x5410);
    reinterpret_cast<uint32_t*>(out + out_pitch)[q] = __byte_perm(a01, a23, 0x7632);
    const uint32_t i01 = __byte_perm(p0, p1, 0x0062), i23 = __byte_perm(p2, p3, 0x0062);    // inf0 inf1 . .
    reinterpret_cast<uint32_t*>(out + 2 * out_pitch)[q] = __byte_perm(i01, i23, 0x5410);
  }
}

// PBHPairing::pairing, src/pbh/pairing.rs:12-47: planes p.x p.y p.inf q.a q.b -> gt.a gt.b
__global__ void __launch_bounds__(kBlock) pairing_kernel(const Tables* __restrict__ gT, size_t n, const uint8_t* __restrict__ in,
                                                          size_t in_pitch, uint8_t* __restrict__ out, size_t out_pitch) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    F32* tag = nullptr;
    G1F<F32> p;
    p.x = f_from_u32(in[i] % 101u, tag); p.y = f_from_u32(in[in_pitch + i] % 101u, tag); p.inf = in[2 * in_pitch + i] != 0;
    const F32 qa = f_from_u32(in[3 * in_pitch + i] % 101u, tag), qb = f_from_u32(in[4 * in_pitch + i] % 101u, tag);
    const GTF<F32> e = pairingf(p, qa, qb, sT.inv101c);
    out[i] = (uint8_t)f_canon101(e.a); out[out_pitch + i] = (uint8_t)f_canon101(e.b);
  }
}

// GTP * GTP (src/pbh/gt.rs:61-69; OP 0: planes a1 b1 a2 b2 -> a b) and GTP::pow(600) (src/pbh/gt.rs:33-59, the final
// exponentiation of src/pbh/pairing.rs:17; OP 1: planes a b -> a b) on the exact FP32 arithmetic of pbh_g1f.cuh
template <int OP>
__global__ void __launch_bounds__(kBlock) gt_kernel(const Tables* __restrict__ gT, size_t n, const uint8_t* __restrict__ in, size_t in_pitch,
                                                     uint8_t* __restrict__ out, size_t out_pitch) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    F32* tag = nullptr;
    GTF<F32> p, r;
    p.a = f_from_u32(in[i] % 101u, tag); p.b = f_from_u32(in[in_pitch + i] % 101u, tag);
    if (OP == 0) {
      GTF<F32> q;
      q.a = f_from_u32(in[2 * in_pitch + i] % 101u, tag); q.b = f_from_u32(in[3 * in_pitch + i] % 101u, tag);
      r = gtf_mul(p, q);
    } else {
      r = gtf_final_exp(p, sT.inv101c);
    }
    out[i] = (uint8_t)f_canon101(r.a); out[out_pitch + i] = (uint8_t)f_canon101(r.b);
  }
}

// Poly / Poly -> (q, r) for ANY divisor (src/poly.rs:230-247), one item per thread: `ln` numerator planes, `ld` divisor
// planes (zero padded; the normalised lengths are implied by the values), ln quotient planes and ld remainder planes out.
// The reference inverts the divisor's leading coefficient at every step and panics on the zero polynomial
// (`lead_d.inv().unwrap()`): status 1, outputs zero.  ln <= 32, ld <= 16.
__global__ void __launch_bounds__(kBlock) poly_divrem_kernel(const Tables* __restrict__ gT, size_t n, uint32_t ln, uint32_t ld,
                                                              const uint8_t* __restrict__ num, size_t num_pitch, const uint8_t* __restrict__ den,
                                                              size_t den_pitch, uint8_t* __restrict__ q, size_t q_pitch, uint8_t* __restrict__ r,
                                                              size_t r_pitch, uint8_t* __restrict__ status) {
  __shared__ uint8_t s_inv[32];
  if (threadIdx.x < 32) s_inv[threadIdx.x] = gT->inv17[threadIdx.x];
  __syncthreads();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t rem[32], d[16], quo[32];
    uint32_t dlen = 0;                                           // normalised length of the divisor (0: the zero polynomial)
    bool num_zero = true;
    for (uint32_t k = 0; k < 32; k++) { rem[k] = k < ln ? mod17(num[(size_t)k * num_pitch + i]) : 0u; quo[k] = 0u; num_zero = num_zero && rem[k] == 0u; }
    for (uint32_t k = 0; k < 16; k++) { d[k] = k < ld ? mod17(den[(size_t)k * den_pitch + i]) : 0u; if (d[k]) dlen = k + 1; }
    // `while !r.is_zero() && r.degree() >= rhs.degree()`: a zero numerator never reaches the inversion, so 0 / 0 = (0, 0)
    const bool panic = dlen == 0 && !num_zero;
    if (dlen != 0) {
      const uint32_t linv = s_inv[d[dlen - 1]];
      for (int top = (int)ln - 1; top >= (int)dlen - 1; top--) {   // r.degree() >= rhs.degree()
        const uint32_t c = mul17(rem[top], linv);
        if (c == 0u) continue;
        quo[top - (dlen - 1)] = c;
        for (uint32_t j = 0; j < dlen; j++) rem[top - j] = mod17(rem[top - j] + 17u * 16u - c * d[dlen - 1 - j]);
      }
    }
    for (uint32_t k = 0; k < ln; k++) q[(size_t)k * q_pitch + i] = (uint8_t)(panic ? 0u : quo[k]);
    for (uint32_t k = 0; k < ld; k++) r[(size_t)k * r_pitch + i] = (uint8_t)(panic ? 0u : rem[k]);
    status[i] = panic ? 1 : 0;
  }
}

// `a += b` / `a -= b` for operands of DIFFERENT lengths exactly as the reference does it (src/poly.rs:165-176, 192-203):
// la and lb planes, zero padded; with len(a) the normalised length of a (the zero polynomial keeps one coefficient),
// out[n] = a[n] +- b[n] below len(a) and b[n] AS IT IS at or beyond it - for the subtraction too, which is quirk Q1.
__global__ void __launch_bounds__(kBlock) poly_addsub_ragged_kernel(size_t n, uint32_t la, uint32_t lb, int subtract, const uint8_t* __restrict__ a,
                                                                     size_t a_pitch, const uint8_t* __restrict__ b, size_t b_pitch,
                                                                     uint8_t* __restrict__ out, size_t out_pitch) {
  const uint32_t lo = la > lb ? la : lb;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t alen = 1;
    for (uint32_t k = 0; k < la; k++) if (mod17(a[(size_t)k * a_pitch + i])) alen = k + 1;
    for (uint32_t k = 0; k < lo; k++) {
      const uint32_t x = k < la ? mod17(a[(size_t)k * a_pitch + i]) : 0u, y = k < lb ? mod17(b[(size_t)k * b_pitch + i]) : 0u;
      out[(size_t)k * out_pitch + i] = (uint8_t)(k < alen ? (subtract ? sub17(x, y) : add17(x, y)) : y);
    }
  }
}

// ---- record <-> plane transposes (include/pbh_b200.h "record wire format") ------------------------------------------
// One thread per 32-byte record: two 128-bit accesses on the record side (a warp touches 1 KB contiguously), byte-wide
// coalesced accesses on the plane side.
__device__ __forceinline__ void load_record(const void* rec, size_t i, uint32_t (&wv)[8]) {
  const uint4* p = reinterpret_cast<const uint4*>(rec) + 2 * i;
  uint4 lo = p[0], hi = p[1];
  wv[0] = lo.x; wv[1] = lo.y; wv[2] = lo.z; wv[3] = lo.w; wv[4] = hi.x; wv[5] = hi.y; wv[6] = hi.z; wv[7] = hi.w;
}
__device__ __forceinline__ uint32_t record_byte(const uint32_t (&wv)[8], int k) { return (wv[k >> 2] >> (8 * (k & 3))) & 0xFFu; }

__global__ void __launch_bounds__(kBlock) witness_records_to_planes_kernel(size_t n, const pbh_witness_record* __restrict__ rec,
                                                                            uint8_t* __restrict__ wit, size_t wit_pitch,
                                                                            uint8_t* __restrict__ rnd, size_t rand_pitch,
                                                                            uint8_t* __restrict__ chal, size_t chal_pitch,
                                                                            uint8_t* __restrict__ u) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t wv[8];
    load_record(rec, i, wv);
    if (wit) {
#pragma unroll
      for (int k = 0; k < 12; k++) wit[(size_t)k * wit_pitch + i] = (uint8_t)record_byte(wv, k);
    }
    if (rnd) {
#pragma unroll
      for (int k = 0; k < 9; k++) rnd[(size_t)k * rand_pitch + i] = (uint8_t)record_byte(wv, 12 + k);
    }
    if (chal) {
#pragma unroll
      for (int k = 0; k < 5; k++) chal[(size_t)k * chal_pitch + i] = (uint8_t)record_byte(wv, 21 + k);
    }
    if (u) u[i] = (uint8_t)record_byte(wv, 26);
  }
}
__global__ void __launch_bounds__(kBlock) proof_records_to_planes_kernel(size_t n, const pbh_proof_record* __restrict__ rec,
                                                                          uint8_t* __restrict__ proof, size_t proof_pitch,
                                                                          uint8_t* __restrict__ status) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t wv[8];
    load_record(rec, i, wv);
    if (proof) {
#pragma unroll
      for (int k = 0; k < 27; k++) proof[(size_t)k * proof_pitch + i] = (uint8_t)record_byte(wv, k);
    }
    if (status) status[i] = (uint8_t)record_byte(wv, 27);
  }
}
__global__ void __launch_bounds__(kBlock) proof_planes_to_records_kernel(size_t n, const uint8_t* __restrict__ proof, size_t proof_pitch,
                                                                          const uint8_t* __restrict__ status,
                                                                          pbh_proof_record* __restrict__ rec) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t wv[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 27; k++) wv[k >> 2] |= (uint32_t)proof[(size_t)k * proof_pitch + i] << (8 * (k & 3));
    if (status) wv[6] |= (uint32_t)status[i] << 24;
    uint4* p = reinterpret_cast<uint4*>(rec) + 2 * i;
    p[0] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
    p[1] = make_uint4(wv[4], wv[5], wv[6], wv[7]);
  }
}

// Peer-window publication for the paths whose summaries come from a separate kernel (unaligned batches): copies `bytes`
// bytes at `src` to the same offset of every peer's window.
__global__ void __launch_bounds__(kBlock) window_publish_kernel(const uint8_t* __restrict__ src, size_t bytes, const PeerWindow PW) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < bytes; i += (size_t)gridDim.x * blockDim.x) {
    const uint8_t v = src[i];
#pragma unroll
    for (uint32_t p = 0; p < 7; p++)
      if (p < PW.n) const_cast<uint8_t*>(src)[(long long)i + PW.delta[p]] = v;
  }
}

// ---- shard summaries ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) pack_verdicts_kernel(size_t n, const uint8_t* __restrict__ result,
                                                                uint8_t* __restrict__ bitmap) {
  const size_t nbytes = (n + 7) / 8;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < nbytes; j += (size_t)gridDim.x * blockDim.x) {
    uint32_t b = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      size_t i = j * 8 + k;
      if (i < n) b |= (uint32_t)(result[i] & 1u) << k;
    }
    bitmap[j] = (uint8_t)b;
  }
}

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// Digest of one item (include/pbh_b200.h, digest_item_* above): two 32-bit lanes seeded with the global item index,
// murmur3-style multiply / rotate rounds over the item's bytes packed four planes per 32-bit word, murmur3 finaliser.
// The batch digest is the sum over items modulo 2^64, so digests of disjoint shards add up to the digest of the whole
// batch (SURVEY.md §8e).
// vec_ok: data and pitch are 4-byte aligned, so a thread takes four consecutive items through one 32-bit word per
// plane (128-byte warp transactions, four independent loads in flight) and transposes 4x4 bytes with PRMT.
__global__ void __launch_bounds__(kBlock) digest_kernel(size_t n, uint64_t first_index, uint32_t planes,
                                                         const uint8_t* __restrict__ data, size_t pitch,
                                                         unsigned long long* __restrict__ out, bool vec_ok) {
  unsigned long long acc = 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t n4 = vec_ok ? n / 4 : 0;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += stride) {
    DigestState h0 = digest_item_begin(first_index + 4 * q, planes), h1 = digest_item_begin(first_index + 4 * q + 1, planes),
                h2 = digest_item_begin(first_index + 4 * q + 2, planes), h3 = digest_item_begin(first_index + 4 * q + 3, planes);
    for (uint32_t k = 0; k < planes; k += 4) {
      uint32_t w0 = reinterpret_cast<const uint32_t*>(data + (size_t)k * pitch)[q];
      uint32_t w1 = k + 1 < planes ? reinterpret_cast<const uint32_t*>(data + (size_t)(k + 1) * pitch)[q] : 0u;
      uint32_t w2 = k + 2 < planes ? reinterpret_cast<const uint32_t*>(data + (size_t)(k + 2) * pitch)[q] : 0u;
      uint32_t w3 = k + 3 < planes ? reinterpret_cast<const uint32_t*>(data + (size_t)(k + 3) * pitch)[q] : 0u;
      uint32_t t0 = __byte_perm(w0, w1, 0x5140), t1 = __byte_perm(w0, w1, 0x7362);
      uint32_t t2 = __byte_perm(w2, w3, 0x5140), t3 = __byte_perm(w2, w3, 0x7362);
      digest_item_word(h0, __byte_perm(t0, t2, 0x5410));
      digest_item_word(h1, __byte_perm(t0, t2, 0x7632));
      digest_item_word(h2, __byte_perm(t1, t3, 0x5410));
      digest_item_word(h3, __byte_perm(t1, t3, 0x7632));
    }
    acc += digest_item_end(h0) + digest_item_end(h1) + digest_item_end(h2) + digest_item_end(h3);
  }
  for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    DigestState h = digest_item_begin(first_index + i, planes);
    for (uint32_t k = 0; k < planes; k += 4) {
      uint32_t wv = 0;
      for (uint32_t b = 0; b < 4 && k + b < planes; b++) wv |= (uint32_t)data[(size_t)(k + b) * pitch + i] << (8 * b);
      digest_item_word(h, wv);
    }
    acc += digest_item_end(h);
  }
  digest_flush(acc, out);
}

// ---- synthetic inputs (SURVEY.md §8d); mirrors oracle_generate_inputs bit for bit -----------------------
struct GenArgs {
  size_t n; uint64_t first_index, seed; int dist;
  uint8_t* wit; size_t wit_pitch;
  uint8_t* rnd; size_t rand_pitch;
  uint8_t* chal; size_t chal_pitch;
  uint8_t* u; uint8_t* attempt;
  const uint8_t* wtab;   // 289 x 3 solutions of x^2 + y^2 = z^2 in F_17, lexicographic
};
__device__ __forceinline__ uint32_t gen_draw(uint64_t base, uint32_t j, uint32_t range) {
  uint64_t r = splitmix64(base + (uint64_t)j * 0xD1B54A32D192ED03ull);
  return (uint32_t)__umul64hi(r, (uint64_t)range);
}
__global__ void __launch_bounds__(kBlock) generate_kernel(const Consts K, const Tables* __restrict__ gT, const GenArgs A) {
  __shared__ Tables sT;
  stage_tables(sT, gT);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t w[12], r[9], c[5], uu = 0, k = 0;
    for (;; k++) {
      // past PBH_GEN_MAX_ATTEMPTS: attempt 0's draw, reported as attempt 255
      const uint64_t kk = k < PBH_GEN_MAX_ATTEMPTS ? k : 0u;
      uint64_t base = splitmix64(A.seed ^ ((A.first_index + i) * 0x9E3779B97F4A7C15ull) ^ (kk * 0xC2B2AE3D27D4EB4Full));
      const uint8_t* s = A.wtab + 3 * gen_draw(base, 0, 289);
      uint32_t x = s[0], y = s[1], z = s[2];
      uint32_t xx = mod17(x * x), yy = mod17(y * y), zz = mod17(z * z);
      w[0] = x; w[1] = y; w[2] = z; w[3] = xx; w[4] = x; w[5] = y; w[6] = z; w[7] = yy; w[8] = xx; w[9] = yy; w[10] = zz; w[11] = zz;
#pragma unroll
      for (int j = 0; j < 9; j++) r[j] = gen_draw(base, 1 + j, 17);
#pragma unroll
      for (int j = 0; j < 5; j++) c[j] = gen_draw(base, 10 + j, 17);
      uu = gen_draw(base, 15, 17);
      if (A.dist == PBH_DIST_UNIFORM || k == PBH_GEN_MAX_ATTEMPTS) break;
      ProofRegs P;
      uint32_t status = prove_one<ALGO_TABLE>(w, r, c, K, sT, P);
      if (status != 0u) continue;
      uint32_t any_inf = 0;
#pragma unroll
      for (int j = 0; j < 9; j++) any_inf |= (P.pt[j] >> 16) & 1u;
      if (any_inf) continue;                                   // verify would stop at in_curve (Q9)
      uint32_t z2 = mul17(c[3], c[3]);
      if (mul17(z2, z2) == 1u) continue;                       // verify would panic on Z_H(z) = 0 (Q4)
      break;
    }
#pragma unroll
    for (int j = 0; j < 12; j++) A.wit[(size_t)j * A.wit_pitch + i] = (uint8_t)w[j];
#pragma unroll
    for (int j = 0; j < 9; j++) A.rnd[(size_t)j * A.rand_pitch + i] = (uint8_t)r[j];
#pragma unroll
    for (int j = 0; j < 5; j++) A.chal[(size_t)j * A.chal_pitch + i] = (uint8_t)c[j];
    A.u[i] = (uint8_t)uu;
    if (A.attempt) A.attempt[i] = (uint8_t)(k < 255u ? k : 255u);
  }
}

// ---- pipe peaks (SURVEY.md §8d): independent chains, no memory traffic ------------------------------------
// WHICH: 0 IMAD, 1 LOP3+IADD3, 2 half IMAD half ALU, 3 FFMA, 4 HFMA2 (two fp16 lanes per op), 5 IDP.4A (dp4a),
//        6 IMAD.HI, 7 half FFMA half IMAD
template <int WHICH>
__global__ void __launch_bounds__(kBlock) int32_peak_kernel(uint32_t iters, uint32_t seed, uint32_t* sink) {
  uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3u + 1u, a2 = a0 * 5u + 2u, a3 = a0 * 7u + 3u, a4 = a0 * 11u + 4u, a5 = a0 * 13u + 5u,
           a6 = a0 * 17u + 6u, a7 = a0 * 19u + 7u;
  const uint32_t m = seed | 1u, c = seed ^ 0x9E3779B9u;
  if (WHICH == 3 || WHICH == 7) {
    float f0 = (float)(a0 & 255), f1 = (float)(a1 & 255), f2 = (float)(a2 & 255), f3 = (float)(a3 & 255), f4 = (float)(a4 & 255),
          f5 = (float)(a5 & 255), f6 = (float)(a6 & 255), f7 = (float)(a7 & 255);
    const float fm = 0.9999f + (float)(seed & 1u) * 1e-6f, fc = (float)(seed & 3u) * 0.25f;
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int rep = 0; rep < 8; rep++) {
        if (WHICH == 3) {
          f0 = fmaf(f0, fm, fc); f1 = fmaf(f1, fm, fc); f2 = fmaf(f2, fm, fc); f3 = fmaf(f3, fm, fc);
          f4 = fmaf(f4, fm, fc); f5 = fmaf(f5, fm, fc); f6 = fmaf(f6, fm, fc); f7 = fmaf(f7, fm, fc);
        } else {
          f0 = fmaf(f0, fm, fc); a1 = a1 * m + c; f2 = fmaf(f2, fm, fc); a3 = a3 * m + c;
          f4 = fmaf(f4, fm, fc); a5 = a5 * m + c; f6 = fmaf(f6, fm, fc); a7 = a7 * m + c;
        }
      }
    }
    a0 = __float_as_uint(f0) ^ __float_as_uint(f2) ^ __float_as_uint(f4) ^ __float_as_uint(f6);
    if (WHICH == 3) { a1 = __float_as_uint(f1); a3 = __float_as_uint(f3); a5 = __float_as_uint(f5); a7 = __float_as_uint(f7); }
    a2 = a4 = a6 = 0;
  } else if (WHICH == 4) {
    __half2 h0 = __floats2half2_rn((float)(a0 & 7), 1.f), h1 = __floats2half2_rn((float)(a1 & 7), 2.f), h2 = __floats2half2_rn((float)(a2 & 7), 3.f),
            h3 = __floats2half2_rn((float)(a3 & 7), 4.f), h4 = __floats2half2_rn((float)(a4 & 7), 5.f), h5 = __floats2half2_rn((float)(a5 & 7), 6.f),
            h6 = __floats2half2_rn((float)(a6 & 7), 7.f), h7 = __floats2half2_rn((float)(a7 & 7), 8.f);
    const __half2 hm = __floats2half2_rn(0.999f + (float)(seed & 1u) * 1e-3f, 0.998f), hc = __floats2half2_rn((float)(seed & 3u) * 0.25f, 0.5f);
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int rep = 0; rep < 8; rep++) {
        h0 = __hfma2(h0, hm, hc); h1 = __hfma2(h1, hm, hc); h2 = __hfma2(h2, hm, hc); h3 = __hfma2(h3, hm, hc);
        h4 = __hfma2(h4, hm, hc); h5 = __hfma2(h5, hm, hc); h6 = __hfma2(h6, hm, hc); h7 = __hfma2(h7, hm, hc);
      }
    }
    __half2 s = __hadd2(__hadd2(__hadd2(h0, h1), __hadd2(h2, h3)), __hadd2(__hadd2(h4, h5), __hadd2(h6, h7)));
    a0 = *reinterpret_cast<uint32_t*>(&s);
    a1 = a2 = a3 = a4 = a5 = a6 = a7 = 0;
  } else {
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int rep = 0; rep < 8; rep++) {
        if (WHICH == 0) {          // IMAD
          a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
          a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
        } else if (WHICH == 1) {   // LOP3 / IADD3 (ALU pipe)
          a0 = (a0 ^ m) + c; a1 = (a1 ^ m) + c; a2 = (a2 ^ m) + c; a3 = (a3 ^ m) + c;
          a4 = (a4 ^ m) + c; a5 = (a5 ^ m) + c; a6 = (a6 ^ m) + c; a7 = (a7 ^ m) + c;
        } else if (WHICH == 2) {   // half IMAD, half ALU
          a0 = a0 * m + c; a1 = (a1 ^ m) + c; a2 = a2 * m + c; a3 = (a3 ^ m) + c;
          a4 = a4 * m + c; a5 = (a5 ^ m) + c; a6 = a6 * m + c; a7 = (a7 ^ m) + c;
        } else if (WHICH == 5) {   // dp4a
          a0 = __dp4a(a0, m, a0); a1 = __dp4a(a1, m, a1); a2 = __dp4a(a2, m, a2); a3 = __dp4a(a3, m, a3);
          a4 = __dp4a(a4, m, a4); a5 = __dp4a(a5, m, a5); a6 = __dp4a(a6, m, a6); a7 = __dp4a(a7, m, a7);
        } else {                   // IMAD.HI
          a0 = __umulhi(a0, m) + c; a1 = __umulhi(a1, m) + c; a2 = __umulhi(a2, m) + c; a3 = __umulhi(a3, m) + c;
          a4 = __umulhi(a4, m) + c; a5 = __umulhi(a5, m) + c; a6 = __umulhi(a6, m) + c; a7 = __umulhi(a7, m) + c;
        }
      }
    }
  }
  uint32_t r = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
  if (r == 0x12345678u) sink[0] = r;   // keeps the chains alive
}

// shift / logic instruction classes of the SHA-256 transcript kernels, one instruction per chain step.
// WHICH: 0 SHF (funnel shift of two registers), 1 IMAD.WIDE.U32 (64-bit product-accumulate: both halves of a rotation),
//        2 LOP3 (three-register xor), 3 IADD3 (three-register add), 4 PRMT (byte permute)
template <int WHICH>
__global__ void __launch_bounds__(kBlock) shift_peak_kernel(uint32_t iters, uint32_t seed, uint32_t* sink) {
  uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3u + 1u, a2 = a0 * 5u + 2u, a3 = a0 * 7u + 3u, a4 = a0 * 11u + 4u, a5 = a0 * 13u + 5u,
           a6 = a0 * 17u + 6u, a7 = a0 * 19u + 7u;
  const uint32_t m = seed | 0x10001u;
  unsigned long long p0 = a0, p1 = a1, p2 = a2, p3 = a3, p4 = a4, p5 = a5, p6 = a6, p7 = a7;
  for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
    for (int rep = 0; rep < 8; rep++) {
      if (WHICH == 0) {
        a0 = __funnelshift_r(a0, a1, 7); a1 = __funnelshift_r(a1, a2, 7); a2 = __funnelshift_r(a2, a3, 7); a3 = __funnelshift_r(a3, a4, 7);
        a4 = __funnelshift_r(a4, a5, 7); a5 = __funnelshift_r(a5, a6, 7); a6 = __funnelshift_r(a6, a7, 7); a7 = __funnelshift_r(a7, a0, 7);
      } else if (WHICH == 1) {
        p0 = (unsigned long long)(uint32_t)p0 * m + p0; p1 = (unsigned long long)(uint32_t)p1 * m + p1;
        p2 = (unsigned long long)(uint32_t)p2 * m + p2; p3 = (unsigned long long)(uint32_t)p3 * m + p3;
        p4 = (unsigned long long)(uint32_t)p4 * m + p4; p5 = (unsigned long long)(uint32_t)p5 * m + p5;
        p6 = (unsigned long long)(uint32_t)p6 * m + p6; p7 = (unsigned long long)(uint32_t)p7 * m + p7;
      } else if (WHICH == 2) {
        a0 = a0 ^ a1 ^ a2; a1 = a1 ^ a2 ^ a3; a2 = a2 ^ a3 ^ a4; a3 = a3 ^ a4 ^ a5;
        a4 = a4 ^ a5 ^ a6; a5 = a5 ^ a6 ^ a7; a6 = a6 ^ a7 ^ a0; a7 = a7 ^ a0 ^ a1;
      } else if (WHICH == 3) {
        a0 = a0 + a1 + a2; a1 = a1 + a2 + a3; a2 = a2 + a3 + a4; a3 = a3 + a4 + a5;
        a4 = a4 + a5 + a6; a5 = a5 + a6 + a7; a6 = a6 + a7 + a0; a7 = a7 + a0 + a1;
      } else {
        a0 = __byte_perm(a0, a1, 0x6543); a1 = __byte_perm(a1, a2, 0x6543); a2 = __byte_perm(a2, a3, 0x6543); a3 = __byte_perm(a3, a4, 0x6543);
        a4 = __byte_perm(a4, a5, 0x6543); a5 = __byte_perm(a5, a6, 0x6543); a6 = __byte_perm(a6, a7, 0x6543); a7 = __byte_perm(a7, a0, 0x6543);
      }
    }
  }
  uint32_t r = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
  unsigned long long q = p0 ^ p1 ^ p2 ^ p3 ^ p4 ^ p5 ^ p6 ^ p7;
  if ((r ^ (uint32_t)q ^ (uint32_t)(q >> 32)) == 0x12345678u) sink[0] = r;
}

// three distinct register operands per instruction (no constant-bank or immediate operand), the shape of a
// polynomial multiply-accumulate: WHICH 0 = FFMA, 1 = IMAD.  8 accumulators, 4 + 4 varying multiplicands.
template <int WHICH>
__global__ void __launch_bounds__(kBlock) mac3_peak_kernel(uint32_t iters, uint32_t seed, uint32_t* sink) {
  if (WHICH == 0) {
    float x0 = 1.0f + threadIdx.x * 1e-7f, x1 = x0 + 1e-6f, x2 = x0 + 2e-6f, x3 = x0 + 3e-6f;
    float y0 = 1e-3f * (seed & 7), y1 = y0 + 1e-4f, y2 = y0 + 2e-4f, y3 = y0 + 3e-4f;
    float c0 = 0, c1 = 1, c2 = 2, c3 = 3, c4 = 4, c5 = 5, c6 = 6, c7 = 7;
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int rep = 0; rep < 8; rep++) {
        c0 = fmaf(x0, y0, c0); c1 = fmaf(x0, y1, c1); c2 = fmaf(x1, y2, c2); c3 = fmaf(x1, y3, c3);
        c4 = fmaf(x2, y0, c4); c5 = fmaf(x2, y1, c5); c6 = fmaf(x3, y2, c6); c7 = fmaf(x3, y3, c7);
      }
      x0 += c7 * 1e-30f; y0 += c0 * 1e-30f;   // keep the multiplicands loop-variant
    }
    float r = c0 + c1 + c2 + c3 + c4 + c5 + c6 + c7;
    if (r == 12345.678f) sink[0] = 1;
  } else {
    uint32_t x0 = seed + threadIdx.x, y0 = seed ^ 0x55u;
    uint32_t c0 = x0, c1 = x0 * 3u + 1u, c2 = x0 * 5u + 2u, c3 = x0 * 7u + 3u, c4 = y0 | 1u, c5 = y0 * 3u + 5u, c6 = y0 * 5u + 6u, c7 = y0 * 7u + 7u;
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int rep = 0; rep < 8; rep++) {
        // every multiplicand is itself an accumulator of the previous repetition, so that ptxas can neither hoist the
        // products out of the unrolled body nor turn the chain into a multiply by 8 (round 1 measured a folded loop)
        c0 = c4 * c5 + c0; c1 = c5 * c6 + c1; c2 = c6 * c7 + c2; c3 = c7 * c4 + c3;
        c4 = c0 * c1 + c4; c5 = c1 * c2 + c5; c6 = c2 * c3 + c6; c7 = c3 * c0 + c7;
      }
    }
    uint32_t r = c0 ^ c1 ^ c2 ^ c3 ^ c4 ^ c5 ^ c6 ^ c7;
    if (r == 0x12345678u) sink[0] = r;
  }
}

// packed fp32x2 FMA (FFMA2, new on sm_100): three distinct 64-bit register-pair operands per instruction, the shape a
// pair-packed polynomial MAC would have.  WHICH 0: all-pair operands; 1: one operand is a broadcast pair (a, a) built
// from a scalar (the multiplicand of a row of an outer-product MAC).
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
  return d;
}
template <int WHICH>
__global__ void __launch_bounds__(kBlock) ffma2_peak_kernel(uint32_t iters, uint32_t seed, uint32_t* sink) {
  float s0 = 1.0f + threadIdx.x * 1e-7f, s1 = s0 + 1e-6f, s2 = s0 + 2e-6f, s3 = s0 + 3e-6f;
  unsigned long long x0 = pack2(s0, s1), x1 = pack2(s1, s2), x2 = pack2(s2, s3), x3 = pack2(s3, s0);
  float t0 = 1e-3f * (seed & 7);
  unsigned long long y0 = pack2(t0, t0 + 1e-4f), y1 = pack2(t0 + 2e-4f, t0 + 3e-4f), y2 = pack2(t0 + 4e-4f, t0 + 5e-4f), y3 = pack2(t0 + 6e-4f, t0 + 7e-4f);
  unsigned long long c0 = pack2(0, 1), c1 = pack2(2, 3), c2 = pack2(4, 5), c3 = pack2(6, 7), c4 = pack2(8, 9), c5 = pack2(10, 11), c6 = pack2(12, 13),
                     c7 = pack2(14, 15);
  for (uint32_t it = 0; it < iters; it++) {
    if (WHICH == 1) { x0 = pack2(s0, s0); x1 = pack2(s1, s1); x2 = pack2(s2, s2); x3 = pack2(s3, s3); }
#pragma unroll
    for (int rep = 0; rep < 8; rep++) {
      c0 = ffma2(x0, y0, c0); c1 = ffma2(x0, y1, c1); c2 = ffma2(x1, y2, c2); c3 = ffma2(x1, y3, c3);
      c4 = ffma2(x2, y0, c4); c5 = ffma2(x2, y1, c5); c6 = ffma2(x3, y2, c6); c7 = ffma2(x3, y3, c7);
    }
    s0 += __uint_as_float((uint32_t)c7) * 1e-30f; y0 = ffma2(c0, pack2(1e-30f, 1e-30f), y0);
    if (WHICH == 0) x0 = ffma2(c7, pack2(1e-30f, 1e-30f), x0);
  }
  unsigned long long r = c0 ^ c1 ^ c2 ^ c3 ^ c4 ^ c5 ^ c6 ^ c7;
  if (r == 0x123456789ull) sink[0] = 1;
}

}  // namespace pbh
