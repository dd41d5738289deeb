// pbh_multi.cpp — several devices driven from ONE process through the C ABI (include/pbh_b200.h, "multi-device").
//
// SURVEY.md 8(b)/(e): a context-creation entry point that takes a device list, one stream per device, one NCCL
// communicator (ncclCommInitAll), batches split contiguously over the devices, and the only exchange at the end: an
// all-gather of the shards' verdict bitmaps and proof digests.  This file is a host-side composition of single-device
// contexts: every kernel is launched through the public `_dev` entry points of pbh_capi.cu; nothing here computes.
//
// NCCL is loaded at run time (dlopen "libnccl.so.2": the copy torch ships when the caller is a Python process that imported
// torch, the system's otherwise), so the library itself has no link-time dependency on it and single-device users never
// touch it.  There is no fallback for the collective: with more than one device and no NCCL, creation fails.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pbh_b200.h"

namespace {

// the slice of nccl.h this file needs (the ABI of these entry points has been stable since NCCL 2.0)
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;
enum { kNcclUint8 = 1 };
struct Nccl {
  void* lib = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string& err) {
    if (lib) return true;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) { err = std::string("NCCL is needed for more than one device and could not be loaded: ") + dlerror(); return false; }
    CommInitAll = (decltype(CommInitAll))dlsym(lib, "ncclCommInitAll");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
    GroupStart = (decltype(GroupStart))dlsym(lib, "ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))dlsym(lib, "ncclGroupEnd");
    GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!CommInitAll || !CommDestroy || !AllGather || !GroupStart || !GroupEnd || !GetErrorString) { err = "libnccl lacks an entry point"; return false; }
    return true;
  }
};

struct Shard {
  int device = 0;
  pbh_ctx* ctx = nullptr;
  ncclComm_t comm = nullptr;
  uint8_t* buf = nullptr;        // wit 12 | rand 9 | chal 5 | u 1 | proof 27 | status 1 | result 1 planes of pitch `cap`
  uint8_t* summary = nullptr;    // bitmap (cap / 8 bytes) then the 64-bit digest
  uint8_t* gathered = nullptr;   // n_dev summaries
  size_t cap = 0;                // items the buffers hold
  cudaEvent_t t0 = nullptr, t1 = nullptr;
};

}  // namespace

struct pbh_multi {
  std::vector<Shard> shards;
  Nccl nccl;
  std::string last_error;
};

namespace {
std::string g_multi_error;

int mfail(pbh_multi* m, int code, const std::string& msg) {
  if (m) m->last_error = msg; else g_multi_error = msg;
  return code;
}
#define MCUDA(m, expr)                                                                          \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess) return mfail(m, PBH_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)

constexpr size_t kAlign = 256;   // shard boundaries: whole tiles, so every shard keeps the aligned TMA path
size_t shard_items(size_t n, size_t n_dev) { return ((n + n_dev - 1) / n_dev + kAlign - 1) / kAlign * kAlign; }

void free_shard_buffers(Shard& s) {
  if (!s.ctx) return;   // a shard whose context was never created (refused device ordinal) owns nothing
  cudaSetDevice(s.device);
  if (s.buf) cudaFree(s.buf);
  if (s.summary) cudaFree(s.summary);
  if (s.gathered) cudaFree(s.gathered);
  s.buf = s.summary = s.gathered = nullptr;
  s.cap = 0;
}
}  // namespace

// host-pointer calls: shard d takes items [d * per, min(n, (d + 1) * per)) through its device's single-device entry point on its own
// host thread (a context serves one host thread at a time; different contexts are independent)
template <class Call>
static int for_each_shard(pbh_multi* m, size_t n, Call call) {
  const size_t n_dev = m->shards.size(), per = shard_items(n, n_dev);
  std::vector<int> rcs(n_dev, PBH_OK);
  std::vector<std::thread> threads;
  for (size_t d = 0; d < n_dev; d++) {
    const size_t lo = std::min(n, d * per), cnt = std::min(n, lo + per) - lo;
    if (cnt == 0) continue;
    threads.emplace_back([&, d, lo, cnt]() { rcs[d] = call(m->shards[d].ctx, lo, cnt); });
  }
  for (std::thread& t : threads) t.join();
  for (size_t d = 0; d < n_dev; d++)
    if (rcs[d] != PBH_OK) return mfail(m, rcs[d], std::string("device ") + std::to_string(m->shards[d].device) + ": " + pbh_last_error(m->shards[d].ctx));
  return PBH_OK;
}

extern "C" {

int pbh_multi_create(const pbh_circuit* circuit, uint8_t srs_secret, uint32_t srs_n, uint8_t omega_pows, const int* devices, int n_dev,
                     pbh_multi** out) {
  if (!circuit || !out || n_dev < 1 || n_dev > 64) return mfail(nullptr, PBH_ERR_BAD_ARGUMENT, "bad argument");
  *out = nullptr;
  pbh_multi* m = new pbh_multi();
  m->shards.resize(n_dev);
  std::vector<int> devs(n_dev);
  for (int d = 0; d < n_dev; d++) devs[d] = devices ? devices[d] : d;
  for (int d = 0; d < n_dev; d++) {
    m->shards[d].device = devs[d];
    int rc = pbh_ctx_create(circuit, srs_secret, srs_n, omega_pows, devs[d], &m->shards[d].ctx);
    if (rc != PBH_OK) {
      g_multi_error = std::string("device ") + std::to_string(devs[d]) + ": " + pbh_last_error(nullptr);
      pbh_multi_destroy(m);
      return rc;
    }
    cudaSetDevice(devs[d]);
    cudaEventCreate(&m->shards[d].t0);
    cudaEventCreate(&m->shards[d].t1);
  }
  if (n_dev > 1) {
    std::string err;
    if (!m->nccl.load(err)) { g_multi_error = err; pbh_multi_destroy(m); return PBH_ERR_UNSUPPORTED; }
    std::vector<ncclComm_t> comms(n_dev);
    ncclResult_t r = m->nccl.CommInitAll(comms.data(), n_dev, devs.data());
    if (r != 0) { g_multi_error = std::string("ncclCommInitAll: ") + m->nccl.GetErrorString(r); pbh_multi_destroy(m); return PBH_ERR_CUDA; }
    for (int d = 0; d < n_dev; d++) m->shards[d].comm = comms[d];
  }
  *out = m;
  return PBH_OK;
}

void pbh_multi_destroy(pbh_multi* m) {
  if (!m) return;
  for (Shard& s : m->shards) {
    if (s.ctx) pbh_ctx_sync(s.ctx);
    if (s.comm) m->nccl.CommDestroy(s.comm);
    free_shard_buffers(s);
    if (s.t0) cudaEventDestroy(s.t0);
    if (s.t1) cudaEventDestroy(s.t1);
    if (s.ctx) pbh_ctx_destroy(s.ctx);
  }
  delete m;
}

int pbh_multi_device_count(const pbh_multi* m) { return m ? (int)m->shards.size() : PBH_ERR_BAD_ARGUMENT; }
pbh_ctx* pbh_multi_ctx(pbh_multi* m, int i) { return (m && i >= 0 && i < (int)m->shards.size()) ? m->shards[i].ctx : nullptr; }
const char* pbh_multi_last_error(const pbh_multi* m) { return m ? m->last_error.c_str() : g_multi_error.c_str(); }
int pbh_multi_set_algo(pbh_multi* m, int algo) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  for (Shard& s : m->shards) { int rc = pbh_ctx_set_algo(s.ctx, algo); if (rc) return mfail(m, rc, pbh_last_error(s.ctx)); }
  return PBH_OK;
}

int pbh_multi_prove_batch(pbh_multi* m, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                          const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !chal || !proof || !status) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) {
    return pbh_prove_batch(ctx, cnt, wit + lo, wit_pitch, rnd + lo, rand_pitch, chal + lo, chal_pitch, proof + lo, proof_pitch, status + lo);
  });
}

int pbh_multi_verify_batch(pbh_multi* m, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal, size_t chal_pitch,
                           const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!proof || !chal || !u || !result) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) {
    return pbh_verify_batch(ctx, cnt, proof + lo, proof_pitch, chal + lo, chal_pitch, u + lo, result + lo, gt ? gt + lo : nullptr, gt_pitch);
  });
}

int pbh_multi_prove_packed(pbh_multi* m, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!in || !out) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) { return pbh_prove_packed(ctx, cnt, in + lo, out + lo); });
}

int pbh_multi_verify_packed(pbh_multi* m, size_t n, const pbh_packed_proof* proofs, const uint32_t* chal_u, uint8_t* result) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!proofs || !chal_u || !result) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) { return pbh_verify_packed(ctx, cnt, proofs + lo, chal_u + lo, result + lo); });
}

int pbh_multi_prove_fs_batch(pbh_multi* m, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                             uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !proof || !status) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) {
    return pbh_prove_fs_batch(ctx, cnt, wit + lo, wit_pitch, rnd + lo, rand_pitch, proof + lo, proof_pitch, status + lo,
                              chal_out ? chal_out + lo : nullptr, chal_pitch);
  });
}

int pbh_multi_verify_fs_batch(pbh_multi* m, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result, uint8_t* chal_out,
                              size_t chal_pitch, uint8_t* gt, size_t gt_pitch) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!proof || !result) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) {
    return pbh_verify_fs_batch(ctx, cnt, proof + lo, proof_pitch, result + lo, chal_out ? chal_out + lo : nullptr, chal_pitch,
                               gt ? gt + lo : nullptr, gt_pitch);
  });
}

int pbh_multi_prove_fs_packed(pbh_multi* m, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!in || !out) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) {
    return pbh_prove_fs_packed(ctx, cnt, in + lo, out + lo, chal_u_out ? chal_u_out + lo : nullptr);
  });
}

int pbh_multi_verify_fs_packed(pbh_multi* m, size_t n, const pbh_packed_proof* proofs, uint8_t* result) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (n == 0) return PBH_OK;
  if (!proofs || !result) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  return for_each_shard(m, n, [&](pbh_ctx* ctx, size_t lo, size_t cnt) { return pbh_verify_fs_packed(ctx, cnt, proofs + lo, result + lo); });
}

}  // extern "C"

// Per-device planes of the sharded pass in Shard::buf (pitch P = Shard::cap items).
struct ShardPlanes {
  uint8_t *wit, *rnd, *chal, *u, *proof, *status, *result;
  size_t P;
};

// The sharded pass of pbh_multi_prove_verify_sharded and pbh_multi_prove_verify_fs_sharded: sizes the per-device buffers, enqueues
// `shard(ctx, planes, first, cnt, bitmap, digest)` on every device (it generates, proves with the fused digest and verifies with
// the fused bitmap), all-gathers the summaries and reads them back from device 0.
template <class ShardPass>
static int sharded_pass(pbh_multi* m, uint64_t n_total, uint64_t first_index, uint8_t* bitmap_out, uint64_t* digests_out,
                        uint64_t* total_digest_out, uint64_t* accepted_out, float* ms_out, ShardPass shard) {
  if (!m) return PBH_ERR_BAD_ARGUMENT;
  if (!bitmap_out) return mfail(m, PBH_ERR_BAD_ARGUMENT, "null pointer");
  const size_t n_dev = m->shards.size();
  if (n_total == 0) { if (total_digest_out) *total_digest_out = 0; if (accepted_out) *accepted_out = 0; if (ms_out) *ms_out = 0; return PBH_OK; }
  const size_t per = shard_items(n_total, n_dev), sum_bytes = per / 8 + 8;
  // (re)size the per-device buffers
  for (Shard& s : m->shards) {
    if (s.cap >= per) continue;
    free_shard_buffers(s);
    MCUDA(m, cudaSetDevice(s.device));
    MCUDA(m, cudaMalloc(&s.buf, 56 * per));
    MCUDA(m, cudaMalloc(&s.summary, sum_bytes));
    MCUDA(m, cudaMalloc(&s.gathered, n_dev * sum_bytes));
    s.cap = per;
  }
  // enqueue every shard: generate -> prove (+ digest) -> verify (+ bitmap), all asynchronous on the device's stream
  for (size_t d = 0; d < n_dev; d++) {
    Shard& s = m->shards[d];
    const uint64_t lo = std::min<uint64_t>(n_total, (uint64_t)d * per), cnt = std::min<uint64_t>(n_total, lo + per) - lo;
    MCUDA(m, cudaSetDevice(s.device));
    cudaStream_t st = (cudaStream_t)pbh_ctx_stream(s.ctx);
    const size_t P = s.cap;
    const ShardPlanes sp{s.buf, s.buf + 12 * P, s.buf + 21 * P, s.buf + 26 * P, s.buf + 27 * P, s.buf + 54 * P, s.buf + 55 * P, P};
    MCUDA(m, cudaEventRecord(s.t0, st));
    MCUDA(m, cudaMemsetAsync(s.summary, 0, per / 8 + 8, st));
    if (cnt) {
      int rc = shard(s.ctx, sp, first_index + lo, (size_t)cnt, s.summary, (uint64_t*)(s.summary + per / 8));
      if (rc) return mfail(m, rc, std::string("device ") + std::to_string(s.device) + ": " + pbh_last_error(s.ctx));
    }
  }
  // the only exchange: ONE all-gather of the shard summaries (verdict bitmap + digest), grouped over the devices of this process
  if (n_dev > 1) {
    m->nccl.GroupStart();
    for (Shard& s : m->shards) {
      ncclResult_t r = m->nccl.AllGather(s.summary, s.gathered, sum_bytes, kNcclUint8, s.comm, (cudaStream_t)pbh_ctx_stream(s.ctx));
      if (r != 0) { m->nccl.GroupEnd(); return mfail(m, PBH_ERR_CUDA, std::string("ncclAllGather: ") + m->nccl.GetErrorString(r)); }
    }
    ncclResult_t r = m->nccl.GroupEnd();
    if (r != 0) return mfail(m, PBH_ERR_CUDA, std::string("ncclGroupEnd: ") + m->nccl.GetErrorString(r));
  }
  float ms = 0;
  for (Shard& s : m->shards) {
    MCUDA(m, cudaSetDevice(s.device));
    MCUDA(m, cudaEventRecord(s.t1, (cudaStream_t)pbh_ctx_stream(s.ctx)));
  }
  for (Shard& s : m->shards) {
    MCUDA(m, cudaSetDevice(s.device));
    MCUDA(m, cudaEventSynchronize(s.t1));
    float e = 0;
    MCUDA(m, cudaEventElapsedTime(&e, s.t0, s.t1));
    ms = std::max(ms, e);
  }
  // device 0 holds every shard's summary (its own when there is one device)
  Shard& s0 = m->shards[0];
  MCUDA(m, cudaSetDevice(s0.device));
  std::vector<uint8_t> host(n_dev * sum_bytes);
  MCUDA(m, cudaMemcpy(host.data(), n_dev > 1 ? s0.gathered : s0.summary, n_dev * sum_bytes, cudaMemcpyDeviceToHost));
  uint64_t total = 0, accepted = 0;
  for (size_t d = 0; d < n_dev; d++) {
    const uint64_t lo = std::min<uint64_t>(n_total, (uint64_t)d * per), cnt = std::min<uint64_t>(n_total, lo + per) - lo;
    const uint8_t* row = host.data() + d * sum_bytes;
    std::memcpy(bitmap_out + lo / 8, row, (cnt + 7) / 8);
    for (size_t b = 0; b < (cnt + 7) / 8; b++) accepted += (uint64_t)__builtin_popcount(row[b]);
    uint64_t dg;
    std::memcpy(&dg, row + per / 8, 8);
    if (digests_out) digests_out[d] = dg;
    total += dg;
  }
  if (total_digest_out) *total_digest_out = total;
  if (accepted_out) *accepted_out = accepted;
  if (ms_out) *ms_out = ms;
  return PBH_OK;
}


extern "C" {

int pbh_multi_prove_verify_sharded(pbh_multi* m, uint64_t n_total, uint64_t first_index, uint64_t seed, int dist, uint8_t* bitmap_out,
                                   uint64_t* digests_out, uint64_t* total_digest_out, uint64_t* accepted_out, float* ms_out) {
  return sharded_pass(m, n_total, first_index, bitmap_out, digests_out, total_digest_out, accepted_out, ms_out,
                      [&](pbh_ctx* ctx, const ShardPlanes& p, uint64_t first, size_t cnt, uint8_t* bitmap, uint64_t* digest) {
                        int rc = pbh_generate_inputs_dev(ctx, cnt, first, seed, dist, p.wit, p.P, p.rnd, p.P, p.chal, p.P, p.u, nullptr);
                        if (!rc) rc = pbh_prove_digest_batch_dev(ctx, cnt, p.wit, p.P, p.rnd, p.P, p.chal, p.P, p.proof, p.P, p.status, first, digest);
                        if (!rc) rc = pbh_verify_bitmap_batch_dev(ctx, cnt, p.proof, p.P, p.chal, p.P, p.u, p.result, bitmap);
                        return rc;
                      });
}

int pbh_multi_prove_verify_fs_sharded(pbh_multi* m, uint64_t n_total, uint64_t first_index, uint64_t seed, int dist, uint8_t* bitmap_out,
                                      uint64_t* digests_out, uint64_t* total_digest_out, uint64_t* accepted_out, float* ms_out) {
  return sharded_pass(m, n_total, first_index, bitmap_out, digests_out, total_digest_out, accepted_out, ms_out,
                      [&](pbh_ctx* ctx, const ShardPlanes& p, uint64_t first, size_t cnt, uint8_t* bitmap, uint64_t* digest) {
                        // the generated challenge and u planes are not used: the transcript derives them
                        int rc = pbh_generate_inputs_dev(ctx, cnt, first, seed, dist, p.wit, p.P, p.rnd, p.P, p.chal, p.P, p.u, nullptr);
                        if (!rc) rc = pbh_prove_fs_digest_batch_dev(ctx, cnt, p.wit, p.P, p.rnd, p.P, p.proof, p.P, p.status, nullptr, 0, first, digest);
                        if (!rc) rc = pbh_verify_fs_bitmap_batch_dev(ctx, cnt, p.proof, p.P, p.result, bitmap);
                        return rc;
                      });
}

}  // extern "C"
