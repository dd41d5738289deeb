// pbh_capi.cu — the extern "C" boundary of include/pbh_b200.h over the sm_100a kernels.
//
// There is no CPU fallback anywhere in this file: every entry point that computes launches a CUDA kernel on
// the context's device, and context creation fails with PBH_ERR_NO_DEVICE when no device is usable.
#include <cuda.h>
#include <cuda_runtime.h>

#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <initializer_list>
#include <type_traits>
#include <condition_variable>
#include <thread>
#include <vector>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>

#include "pbh_kernels.cuh"
#include "pbh_packed.cuh"
#include "pbh_setup.hpp"

using namespace pbh;

namespace {
std::string g_last_error;
std::mutex g_err_mutex;
void set_global_error(const std::string& e) { std::lock_guard<std::mutex> l(g_err_mutex); g_last_error = e; }
}  // namespace

// Host-pointer entry points: the batch is cut into chunks that cycle through kSlots staging buffers, each with its own
// stream, so the H2D copy of chunk k+2, the kernel of chunk k+1 and the D2H copy of chunk k overlap (PCIe is full duplex).
static constexpr size_t kChunkMax = (size_t)1 << 20;   // upper bound of the staged chunk (staging buffers are sized for it lazily)
static constexpr int kSlots = 4;
static constexpr uint32_t kCounterRing = 4096, kCounterGraphPool = 32768;   // launch-local scheduler records
static constexpr uint32_t kCounterWords = 4;   // {next tile, blocks done, 64-bit digest accumulator}: 16 bytes per launch

// ---- pageable host buffers ----------------------------------------------------------------------------------------------
// A copy between PAGEABLE host memory and the device is staged by the driver through its own page-locked buffer, on the
// calling thread, at ~12 GB/s - a fifth of the link.  The staged entry points therefore do the staging themselves: every
// staging slot has a page-locked MIRROR of its device buffer; inputs are copied into the mirror by a small pool of host
// threads (row segments in parallel) and travel from there with an asynchronous copy, outputs land in the mirror and are
// copied out to the caller's memory by the same pool once the slot's stream has drained (before the slot is reused, and at
// the end of the call).  Page-locked caller memory bypasses all of this.
struct CopyTask { uint8_t* dst; const uint8_t* src; size_t bytes; };
class CopyPool {
 public:
  explicit CopyPool(int workers) {
    for (int i = 0; i < workers; i++) threads_.emplace_back([this] { loop(); });
  }
  ~CopyPool() {
    { std::lock_guard<std::mutex> l(m_); stop_ = true; }
    cv_.notify_all();
    for (std::thread& t : threads_) t.join();
  }
  // runs every task (the caller works too) and returns when all are done
  void run(std::vector<CopyTask>& tasks) {
    if (tasks.empty()) return;
    std::unique_lock<std::mutex> l(m_);
    tasks_.swap(tasks);
    next_ = 0;
    pending_ = tasks_.size();
    cv_.notify_all();
    work(l);
    done_.wait(l, [this] { return pending_ == 0; });
    tasks_.clear();
    next_ = 0;
  }
 private:
  void work(std::unique_lock<std::mutex>& l) {
    while (next_ < tasks_.size()) {
      const CopyTask t = tasks_[next_++];
      l.unlock();
      std::memcpy(t.dst, t.src, t.bytes);
      l.lock();
      if (--pending_ == 0) done_.notify_all();
    }
  }
  void loop() {
    std::unique_lock<std::mutex> l(m_);
    for (;;) {
      cv_.wait(l, [this] { return stop_ || next_ < tasks_.size(); });
      if (stop_) return;
      work(l);
    }
  }
  std::mutex m_;
  std::condition_variable cv_, done_;
  std::vector<CopyTask> tasks_;
  size_t next_ = 0, pending_ = 0;
  bool stop_ = false;
  std::vector<std::thread> threads_;
};

struct pbh_ctx {
  int device = 0;
  int sm_count = 148;
  int algo = PBH_ALGO_TABLE;
  int prover_variant = 0;
  size_t chunk = (size_t)1 << 18;          // items per staged chunk of the host-pointer entry points (PBH_OPT_CHUNK_LOG2)
  bool pbh_circuit = false;                // the context's constants equal the compile-time PbhCK (pbh_prove_f32.cuh)
  int specialise = 1;                      // PBH_OPT_SPECIALISE
  int use_tma = 1;                         // TMA-staged tiles when base/pitch alignment allows (PBH_OPT_TMA)
  int host_direct = 1;                     // PBH_OPT_HOST_DIRECT: run the kernels in place on page-locked, mapped host buffers
  int prover_fp32 = 1;                     // PBH_ALGO_TABLE prover: FP32-pipe arithmetic (1) or the int32 routine (0)
  int verifier_fp32 = 0;                   // PBH_ALGO_TABLE verifier scalars: int32 (0, default: faster since the reductions lost their multiply-high) or FP32 (1)
  HostSetup hs;
  Tables* d_tables = nullptr;
  FixedBaseTables* d_pairs = nullptr;
  uint8_t* d_wtab = nullptr;
  // dynamic tile scheduler: one {next tile, blocks done} pair PER LAUNCH.  Direct launches take pairs round-robin from a ring
  // (a pair is reused only kCounterRing launches later, long after the launch that held it has finished: every host-pointer
  // call synchronises and the last block of a launch resets its pair); launches recorded into a CUDA graph take pairs from a
  // pool that is never reused, because a captured launch replays for as long as the graph lives.
  unsigned int* d_tile_counters = nullptr;
  uint32_t counter_seq = 0, graph_counters_used = 0;
  cudaStream_t compute = nullptr;          // `_dev` entry points
  cudaStream_t slot_stream[kSlots] = {};
  uint8_t* slot_buf[kSlots] = {};
  size_t slot_bytes = 0;
  uint64_t launches = 0;
  uint8_t* slot_mirror[kSlots] = {};       // page-locked mirrors of slot_buf for pageable caller memory (allocated on first use)
  bool slot_dirty[kSlots] = {};            // the slot's mirror is in use by copies in flight (sync before the slot is reused)
  std::vector<CopyTask> slot_out[kSlots];  // copy-outs mirror -> caller memory, due once the slot's stream has drained
  CopyPool* pool = nullptr;
  int host_stage = 1;                      // PBH_OPT_HOST_STAGE: own staging of pageable memory (1) or the driver's (0)
  // PBH_OPT_PROOF_RESIDENT: the packed proofs a lane's prove call has just produced are still on the device (as byte planes, rows
  // 26..52 of the lane buffer) when the verify call for the SAME host buffer follows on the same lane
  int proof_resident = 1;
  const void* resident_host[kSlots] = {};
  size_t resident_n[kSlots] = {};
  uint8_t* lane_buf[kSlots] = {};          // whole-batch staging of the asynchronous lanes (PBH_OPT_LANE_MODE 1 and 3)
  size_t lane_bytes[kSlots] = {};
  int lane_mode = 3;                       // PBH_OPT_LANE_MODE
  int grid_scale = 2;                      // persistent-grid blocks per SM are grid_scale/2 of the kernel's residency (1: half grids, async lanes)
  int numa_node = -1;                      // NUMA node of the device's PCIe root (sysfs), -1 when the platform does not say
  std::map<void*, std::pair<size_t, bool>> host_allocs;   // pbh_host_alloc: pointer -> (bytes, mmap'ed + registered)
  // peer window (pbh_window_*): this rank's copy of the world x bytes_per_rank window and the peers' copies
  uint8_t* win_base = nullptr;
  size_t win_bytes_per_rank = 0;
  int win_rank = 0, win_world = 0;
  bool win_owner = false, win_attached = false;
  uint8_t* win_peer[8] = {};
  bool win_peer_ipc[8] = {};
  std::string last_error;
};

#define CTX_CHECK(ctx)                                     \
  do {                                                     \
    if (!(ctx)) { set_global_error("null context"); return PBH_ERR_BAD_ARGUMENT; } \
    (void)cudaGetLastError(); /* a stale, non-sticky error of an earlier call (say, a refused device ordinal) is not this call's */ \
  } while (0)

#define CUDA_TRY(ctx, expr)                                                                      \
  do {                                                                                           \
    cudaError_t e__ = (expr);                                                                    \
    if (e__ != cudaSuccess) {                                                                    \
      (ctx)->last_error = std::string(#expr) + ": " + cudaGetErrorString(e__);                   \
      return PBH_ERR_CUDA;                                                                       \
    }                                                                                            \
  } while (0)

#define PBH_TRY(expr)              \
  do {                             \
    int rc__ = (expr);             \
    if (rc__ != PBH_OK) return rc__; \
  } while (0)

static int device_numa_node(int device);
static void window_release(pbh_ctx* ctx);

static int fail(pbh_ctx* ctx, int code, const char* msg) {
  if (ctx) ctx->last_error = msg; else set_global_error(msg);
  return code;
}

static int grid_for(const pbh_ctx* ctx, size_t n, int per_sm) {
  size_t blocks = (n + kBlock - 1) / kBlock;
  size_t cap = (size_t)ctx->sm_count * per_sm;   // a multiple of the SM count; blocks loop grid-stride
  return (int)std::max<size_t>(1, std::min(blocks, cap));
}

// Every function below is declared extern "C" by include/pbh_b200.h and inherits that linkage.

void pbh_circuit_pbh_test(pbh_circuit* out) {
  // src/pbh/mod.rs:56-67: three mul gates, one add gate
  const uint8_t m1 = 16;
  const uint8_t ql[4] = {0, 0, 0, 1}, qr[4] = {0, 0, 0, 1}, qo[4] = {m1, m1, m1, m1}, qm[4] = {1, 1, 1, 0}, qc[4] = {0, 0, 0, 0};
  const uint8_t caw[4] = {PBH_COPY_B, PBH_COPY_B, PBH_COPY_B, PBH_COPY_C}, cai[4] = {1, 2, 3, 1};
  const uint8_t cbw[4] = {PBH_COPY_A, PBH_COPY_A, PBH_COPY_A, PBH_COPY_C}, cbi[4] = {1, 2, 3, 2};
  const uint8_t ccw[4] = {PBH_COPY_A, PBH_COPY_B, PBH_COPY_C, PBH_COPY_C}, cci[4] = {4, 4, 4, 3};
  for (int i = 0; i < 4; i++) {
    out->q_l[i] = ql[i]; out->q_r[i] = qr[i]; out->q_o[i] = qo[i]; out->q_m[i] = qm[i]; out->q_c[i] = qc[i];
    out->c_a_wire[i] = caw[i]; out->c_a_index[i] = cai[i];
    out->c_b_wire[i] = cbw[i]; out->c_b_index[i] = cbi[i];
    out->c_c_wire[i] = ccw[i]; out->c_c_index[i] = cci[i];
  }
}

int pbh_ctx_create(const pbh_circuit* circuit, uint8_t srs_secret, uint32_t srs_n, uint8_t omega_pows, int device,
                   pbh_ctx** out) {
  if (!circuit || !out) return fail(nullptr, PBH_ERR_BAD_ARGUMENT, "null argument");
  *out = nullptr;
  pbh_ctx* ctx = new pbh_ctx();
  std::string err;
  int rc = host_setup(*circuit, srs_secret, srs_n, omega_pows, ctx->hs, err);
  if (rc != PBH_OK) { set_global_error(err); delete ctx; return rc; }
  ctx->pbh_circuit = consts_match_pbh(ctx->hs.KF, ctx->hs.K.n_pts);

  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    set_global_error(std::string("no usable CUDA device (there is no CPU fallback): ") +
                     (ce != cudaSuccess ? cudaGetErrorString(ce) : "device index out of range"));
    delete ctx;
    return PBH_ERR_NO_DEVICE;
  }
  ctx->device = device;
  auto bail = [&](const char* what, cudaError_t e) {
    set_global_error(std::string(what) + ": " + cudaGetErrorString(e));
    pbh_ctx_destroy(ctx);
    return PBH_ERR_CUDA;
  };
  if ((ce = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", ce);
  cudaDeviceProp prop;
  if ((ce = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", ce);
  ctx->sm_count = prop.multiProcessorCount;
  ctx->numa_node = device_numa_node(device);
  if ((ce = cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", ce);
  for (int s = 0; s < kSlots; s++)
    if ((ce = cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", ce);
  if ((ce = cudaMalloc(&ctx->d_pairs, sizeof(FixedBaseTables))) != cudaSuccess) return bail("cudaMalloc(pair tables)", ce);
  if ((ce = cudaMemcpy(ctx->d_pairs, &ctx->hs.P, sizeof(FixedBaseTables), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy(pair tables)", ce);
  if ((ce = cudaMalloc(&ctx->d_tables, sizeof(Tables))) != cudaSuccess) return bail("cudaMalloc(tables)", ce);
  {
    Tables dev_copy = ctx->hs.T;          // the device copy points at the device pair tables, the host copy at the host ones
    dev_copy.fixed = ctx->d_pairs;
    if ((ce = cudaMemcpy(ctx->d_tables, &dev_copy, sizeof(Tables), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy(tables)", ce);
  }
  // witness table of the synthetic-input generator: solutions of x^2 + y^2 = z^2 in F_17^3, lexicographic
  uint8_t wtab[289 * 3];
  int nw = 0;
  for (int x = 0; x < 17; x++)
    for (int y = 0; y < 17; y++)
      for (int z = 0; z < 17; z++)
        if ((x * x + y * y) % 17 == (z * z) % 17) { wtab[3 * nw] = x; wtab[3 * nw + 1] = y; wtab[3 * nw + 2] = z; nw++; }
  if ((ce = cudaMalloc(&ctx->d_tile_counters, (kCounterRing + kCounterGraphPool) * kCounterWords * sizeof(unsigned int))) != cudaSuccess) return bail("cudaMalloc(counters)", ce);
  if ((ce = cudaMemset(ctx->d_tile_counters, 0, (kCounterRing + kCounterGraphPool) * kCounterWords * sizeof(unsigned int))) != cudaSuccess) return bail("cudaMemset(counters)", ce);
  if ((ce = cudaMalloc(&ctx->d_wtab, sizeof(wtab))) != cudaSuccess) return bail("cudaMalloc(wtab)", ce);
  if ((ce = cudaMemcpy(ctx->d_wtab, wtab, sizeof(wtab), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy(wtab)", ce);
  *out = ctx;
  return PBH_OK;
}

void pbh_ctx_destroy(pbh_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (int s = 0; s < kSlots; s++) {
    if (ctx->slot_stream[s]) { cudaStreamSynchronize(ctx->slot_stream[s]); cudaStreamDestroy(ctx->slot_stream[s]); }
    if (ctx->slot_buf[s]) cudaFree(ctx->slot_buf[s]);
    if (ctx->lane_buf[s]) cudaFree(ctx->lane_buf[s]);
  }
  if (ctx->compute) { cudaStreamSynchronize(ctx->compute); cudaStreamDestroy(ctx->compute); }
  for (auto& a : ctx->host_allocs) { if (a.second.second) { cudaHostUnregister(a.first); munmap(a.first, a.second.first); } else cudaFreeHost(a.first); }
  ctx->host_allocs.clear();
  if (ctx->d_tables) cudaFree(ctx->d_tables);
  if (ctx->d_pairs) cudaFree(ctx->d_pairs);
  if (ctx->d_wtab) cudaFree(ctx->d_wtab);
  window_release(ctx);
  delete ctx->pool;
  ctx->pool = nullptr;
  for (int s = 0; s < kSlots; s++)
    if (ctx->slot_mirror[s]) { cudaFreeHost(ctx->slot_mirror[s]); ctx->slot_mirror[s] = nullptr; }
  if (ctx->d_tile_counters) cudaFree(ctx->d_tile_counters);
  delete ctx;
}

const char* pbh_last_error(const pbh_ctx* ctx) {
  if (ctx) return ctx->last_error.c_str();
  std::lock_guard<std::mutex> l(g_err_mutex);
  static thread_local std::string copy;
  copy = g_last_error;
  return copy.c_str();
}

int pbh_ctx_set_algo(pbh_ctx* ctx, int algo) {
  CTX_CHECK(ctx);
  if (algo != PBH_ALGO_ARITH && algo != PBH_ALGO_TABLE) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "unknown algo");
  ctx->algo = algo;
  return PBH_OK;
}
int pbh_ctx_get_algo(const pbh_ctx* ctx) { return ctx ? ctx->algo : PBH_ERR_BAD_ARGUMENT; }
int pbh_ctx_set_option(pbh_ctx* ctx, int option, int value) {
  CTX_CHECK(ctx);
  if (option == PBH_OPT_PROVER_FP32) { ctx->prover_fp32 = value != 0; return PBH_OK; }
  if (option == PBH_OPT_PROVER_LAUNCH_SHAPE) { ctx->prover_variant = value; return PBH_OK; }
  if (option == PBH_OPT_TMA) { ctx->use_tma = value != 0; return PBH_OK; }
  if (option == PBH_OPT_SPECIALISE) { ctx->specialise = value != 0; return PBH_OK; }
  if (option == PBH_OPT_HOST_DIRECT) { ctx->host_direct = value != 0; return PBH_OK; }
  if (option == PBH_OPT_VERIFIER_FP32) { ctx->verifier_fp32 = value != 0; return PBH_OK; }
  if (option == PBH_OPT_LANE_MODE) {
    if (value != 0 && value != 1 && value != 3) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "lane mode must be 0, 1 or 3");
    ctx->lane_mode = value;
    return PBH_OK;
  }
  if (option == PBH_OPT_HOST_STAGE) { ctx->host_stage = value != 0; return PBH_OK; }
  if (option == PBH_OPT_PROOF_RESIDENT) {
    ctx->proof_resident = value != 0;
    for (int s = 0; s < kSlots; s++) ctx->resident_host[s] = nullptr;
    return PBH_OK;
  }
  if (option == PBH_OPT_CHUNK_LOG2) {
    if (value < 8 || value > 20) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "chunk log2 must be in [8, 20]");
    ctx->chunk = (size_t)1 << value;
    return PBH_OK;
  }
  return fail(ctx, PBH_ERR_BAD_ARGUMENT, "unknown option");
}
int pbh_ctx_device(const pbh_ctx* ctx) { return ctx ? ctx->device : PBH_ERR_BAD_ARGUMENT; }
void* pbh_ctx_stream(pbh_ctx* ctx) { return ctx ? (void*)ctx->compute : nullptr; }
uint64_t pbh_ctx_launch_count(const pbh_ctx* ctx) { return ctx ? ctx->launches : 0; }

int pbh_ctx_sync(pbh_ctx* ctx) {
  CTX_CHECK(ctx);
  for (int s = 0; s < kSlots; s++) ctx->resident_host[s] = nullptr;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute));
  for (int s = 0; s < kSlots; s++) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot_stream[s]));
  return PBH_OK;
}

int pbh_ctx_get_srs(const pbh_ctx* ctx, uint8_t* g1s_xy_inf, size_t cap_points, uint32_t* n_points, uint8_t g2[4]) {
  if (!ctx) return PBH_ERR_BAD_ARGUMENT;
  if (n_points) *n_points = (uint32_t)ctx->hs.g1s.size();
  if (g1s_xy_inf) {
    for (size_t i = 0; i < ctx->hs.g1s.size() && i < cap_points; i++) {
      g1s_xy_inf[3 * i] = (uint8_t)ctx->hs.g1s[i].x; g1s_xy_inf[3 * i + 1] = (uint8_t)ctx->hs.g1s[i].y;
      g1s_xy_inf[3 * i + 2] = (uint8_t)ctx->hs.g1s[i].inf;
    }
  }
  if (g2) { g2[0] = (uint8_t)ctx->hs.g2_1[0]; g2[1] = (uint8_t)ctx->hs.g2_1[1]; g2[2] = (uint8_t)ctx->hs.g2_s[0]; g2[3] = (uint8_t)ctx->hs.g2_s[1]; }
  return PBH_OK;
}

int pbh_ctx_get_verifier_constants(const pbh_ctx* ctx, uint8_t c[24]) {
  if (!ctx || !c) return PBH_ERR_BAD_ARGUMENT;
  for (int j = 0; j < 8; j++) {
    c[3 * j] = (uint8_t)ctx->hs.vconst[j].x; c[3 * j + 1] = (uint8_t)ctx->hs.vconst[j].y; c[3 * j + 2] = (uint8_t)ctx->hs.vconst[j].inf;
  }
  return PBH_OK;
}

// The {next tile, blocks done, digest accumulator} record of the launch about to be enqueued on `st`: launch-local, zero when
// the launch starts (the last block of the previous holder reset it).  nullptr when a capturing stream has used up the graph pool.
static unsigned int* fresh_tile_counter(pbh_ctx* ctx, cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
  if (cap != cudaStreamCaptureStatusNone) {
    if (ctx->graph_counters_used >= kCounterGraphPool) return nullptr;
    return ctx->d_tile_counters + (size_t)(kCounterRing + ctx->graph_counters_used++) * kCounterWords;
  }
  return ctx->d_tile_counters + (size_t)(ctx->counter_seq++ % kCounterRing) * kCounterWords;
}

// ---- TMA tensor maps --------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled is a driver entry point; it is resolved through the runtime so that the library does not
// link against libcuda directly.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      return nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// a (n items x planes) byte-plane batch as a 2-D u8 tensor with box (kTile, planes); false when TMA cannot address it
static bool make_plane_map(CUtensorMap* map, const void* base, size_t n, size_t pitch, uint32_t planes) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || n == 0 || n >= ((size_t)1 << 31) || ((uintptr_t)base % 16) != 0 || (pitch % 16) != 0) return false;
  cuuint64_t dims[2] = {(cuuint64_t)n, planes};
  cuuint64_t strides[1] = {(cuuint64_t)pitch};
  cuuint32_t box[2] = {(cuuint32_t)kTile, planes};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ---- device-pointer entry points -----------------------------------------------------------------------
static int launch_digest(pbh_ctx* ctx, cudaStream_t st, size_t n, uint64_t first_index, uint32_t planes, const uint8_t* data,
                         size_t pitch, uint64_t* out) {
  const bool vec_ok = ((uintptr_t)data % 4 == 0) && (pitch % 4 == 0);
  digest_kernel<<<grid_for(ctx, vec_ok ? (n + 3) / 4 : n, 8), kBlock, 0, st>>>(n, first_index, planes, data, pitch,
                                                                             (unsigned long long*)out, vec_ok);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}

// The peers of a summary pointer: non-empty when the context has an attached peer window and [p, p + bytes) lies inside this
// rank's region of it.
static PeerWindow peer_window_for(const pbh_ctx* ctx, const void* p, size_t bytes) {
  PeerWindow pw{};
  if (!ctx->win_attached || !p) return pw;
  static const bool no_push = std::getenv("PBH_DEBUG_WINDOW_NO_PUSH") != nullptr;   // diagnostic: what do the remote stores cost?
  if (no_push) return pw;
  const uint8_t* lo = ctx->win_base + (size_t)ctx->win_rank * ctx->win_bytes_per_rank;
  const uint8_t* q = static_cast<const uint8_t*>(p);
  if (q < lo || q + bytes > lo + ctx->win_bytes_per_rank) return pw;
  for (int r = 0; r < ctx->win_world; r++) {
    if (r == ctx->win_rank || !ctx->win_peer[r]) continue;
    pw.delta[pw.n++] = (long long)(ctx->win_peer[r] - ctx->win_base);
  }
  return pw;
}
static int launch_publish(pbh_ctx* ctx, cudaStream_t st, const void* src, size_t bytes, const PeerWindow& pw) {
  if (pw.n == 0 || bytes == 0) return PBH_OK;
  window_publish_kernel<<<(int)std::max<size_t>(1, std::min<size_t>((bytes + kBlock - 1) / kBlock, 64)), kBlock, 0, st>>>(
      static_cast<const uint8_t*>(src), bytes, pw);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}

// digest (nullable): device uint64, already zeroed on `st`; receives the digest of the 27 proof planes
static int launch_prove(pbh_ctx* ctx, cudaStream_t st, const ProveArgs& A, uint64_t first_index = 0, uint64_t* digest = nullptr) {
  if (A.n == 0) return PBH_OK;
  if (ctx->prover_fp32 && ctx->use_tma) {
    ProveTmaMaps M;
    if (make_plane_map(&M.wit, A.wit, A.n, A.wit_pitch, 12) && make_plane_map(&M.rnd, A.rnd, A.n, A.rand_pitch, 9) &&
        make_plane_map(&M.chal, A.chal, A.n, A.chal_pitch, 5) && make_plane_map(&M.proof, A.proof, A.n, A.proof_pitch, 27)) {
      size_t tiles = (A.n + kTile - 1) / kTile;
      int grid = (int)std::min<size_t>(tiles, (size_t)ctx->sm_count * ctx->grid_scale);   // persistent: two resident blocks per SM (one on the async lanes)
      unsigned int* tc = fresh_tile_counter(ctx, st);
      if (!tc) return fail(ctx, PBH_ERR_UNSUPPORTED, "too many launches captured into CUDA graphs from this context");
      unsigned long long* dg = (unsigned long long*)digest;
      const PeerWindow pw = peer_window_for(ctx, digest, sizeof(uint64_t));
      // the compile-time instantiation for the reference's own circuit + SRS(2, 6) when the context's constants match it
      const bool special = ctx->pbh_circuit && ctx->specialise;
      if (ctx->algo == PBH_ALGO_TABLE && special)
        prove_f32_tma_kernel<ALGO_TABLE, true><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, ctx->d_tables, A.proof, A.proof_pitch, A.status, A.n, first_index, dg, tc, pw);
      else if (ctx->algo == PBH_ALGO_TABLE)
        prove_f32_tma_kernel<ALGO_TABLE, false><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, ctx->d_tables, A.proof, A.proof_pitch, A.status, A.n, first_index, dg, tc, pw);
      else if (special)
        prove_f32_tma_kernel<ALGO_ARITH, true><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, ctx->d_tables, A.proof, A.proof_pitch, A.status, A.n, first_index, dg, tc, pw);
      else
        prove_f32_tma_kernel<ALGO_ARITH, false><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, ctx->d_tables, A.proof, A.proof_pitch, A.status, A.n, first_index, dg, tc, pw);
      ctx->launches++;
      CUDA_TRY(ctx, cudaGetLastError());
      return PBH_OK;
    }
    // base or pitch not 16-byte aligned: fall through to the plain-load kernel
  }
  int grid = grid_for(ctx, A.n, 8);
  if (ctx->prover_fp32 && ctx->algo == PBH_ALGO_ARITH) {
    prove_f32_kernel<ALGO_ARITH, 256, 2><<<grid_for(ctx, A.n, 8), 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->d_tables, A);
  } else if (ctx->prover_fp32) {
    // launch shape of the FP32 prover: threads per block / resident blocks per SM the register budget is capped for
    switch (ctx->prover_variant) {
      case 1: prove_f32_kernel<ALGO_TABLE, 256, 1><<<grid_for(ctx, A.n, 8), 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->d_tables, A); break;
      case 2: prove_f32_kernel<ALGO_TABLE, 128, 4><<<(int)std::max<size_t>(1, std::min((A.n + 127) / 128, (size_t)ctx->sm_count * 16)), 128, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->d_tables, A); break;
      case 3: prove_f32_kernel<ALGO_TABLE, 128, 5><<<(int)std::max<size_t>(1, std::min((A.n + 127) / 128, (size_t)ctx->sm_count * 20)), 128, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->d_tables, A); break;
      case 4: prove_f32_kernel<ALGO_TABLE, 128, 6><<<(int)std::max<size_t>(1, std::min((A.n + 127) / 128, (size_t)ctx->sm_count * 24)), 128, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->d_tables, A); break;
      default: prove_f32_kernel<ALGO_TABLE, 256, 2><<<grid_for(ctx, A.n, 8), 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->d_tables, A); break;
    }
  } else if (ctx->algo == PBH_ALGO_TABLE) prove_kernel<ALGO_TABLE><<<grid, kBlock, 0, st>>>(ctx->hs.K, ctx->d_tables, A);
  else prove_kernel<ALGO_ARITH><<<grid, kBlock, 0, st>>>(ctx->hs.K, ctx->d_tables, A);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  if (digest) {   // not fused on this path: the digest kernel accumulates into a zeroed word
    CUDA_TRY(ctx, cudaMemsetAsync(digest, 0, sizeof(uint64_t), st));
    int rc = launch_digest(ctx, st, A.n, first_index, 27, A.proof, A.proof_pitch, digest);
    if (rc) return rc;
    return launch_publish(ctx, st, digest, sizeof(uint64_t), peer_window_for(ctx, digest, sizeof(uint64_t)));
  }
  return PBH_OK;
}
static int launch_verify(pbh_ctx* ctx, cudaStream_t st, const VerifyArgs& A_in) {
  if (A_in.n == 0) return PBH_OK;
  VerifyArgs A = A_in;
  const PeerWindow pw = peer_window_for(ctx, A_in.bitmap, (A_in.n + 7) / 8);
  uint8_t* bitmap_later = nullptr;
  if (A.bitmap && (((uintptr_t)A.bitmap % 4) != 0)) { bitmap_later = A.bitmap; A.bitmap = nullptr; }
  if (ctx->use_tma) {
    VerifyTmaMaps M;
    if (make_plane_map(&M.proof, A.proof, A.n, A.proof_pitch, 27) && make_plane_map(&M.chal, A.chal, A.n, A.chal_pitch, 5) &&
        make_plane_map(&M.u, A.u, A.n, (A.n + 15) / 16 * 16, 1)) {
      size_t tiles = (A.n + kTile - 1) / kTile;
      unsigned int* tc = fresh_tile_counter(ctx, st);
      if (!tc) return fail(ctx, PBH_ERR_UNSUPPORTED, "too many launches captured into CUDA graphs from this context");
      if (ctx->algo == PBH_ALGO_TABLE) {
        int grid = (int)std::min<size_t>(tiles, (size_t)ctx->sm_count * 2 * ctx->grid_scale);
        if (A.bitmap && pw.n) verify_tma_kernel<ALGO_TABLE, 4, true><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, ctx->verifier_fp32 != 0, ctx->d_tables, A, tc, pw);
        else verify_tma_kernel<ALGO_TABLE, 4, false><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, ctx->verifier_fp32 != 0, ctx->d_tables, A, tc, PeerWindow{});
      } else {
        int grid = (int)std::min<size_t>(tiles, (size_t)ctx->sm_count * (ctx->grid_scale == 2 ? 3 : 2));
        if (A.bitmap && pw.n) verify_tma_kernel<ALGO_ARITH, 3, true><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, false, ctx->d_tables, A, tc, pw);
        else verify_tma_kernel<ALGO_ARITH, 3, false><<<grid, kTile, 0, st>>>(M, ctx->hs.K, ctx->hs.KF, false, ctx->d_tables, A, tc, PeerWindow{});
      }
      ctx->launches++;
      CUDA_TRY(ctx, cudaGetLastError());
      if (bitmap_later) {
        pack_verdicts_kernel<<<grid_for(ctx, (A.n + 7) / 8, 8), kBlock, 0, st>>>(A.n, A.result, bitmap_later);
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
        return launch_publish(ctx, st, bitmap_later, (A.n + 7) / 8, pw);
      }
      return PBH_OK;
    }
  }
  if (A.bitmap) { bitmap_later = A.bitmap; A.bitmap = nullptr; }   // the plain kernels do not pack
  int grid = grid_for(ctx, A.n, 8);
  if (ctx->algo == PBH_ALGO_TABLE) verify_kernel<ALGO_TABLE><<<grid, kBlock, 0, st>>>(ctx->hs.K, ctx->hs.KF, ctx->verifier_fp32 != 0, ctx->d_tables, A);
  else verify_kernel<ALGO_ARITH><<<grid, kBlock, 0, st>>>(ctx->hs.K, ctx->hs.KF, false, ctx->d_tables, A);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  if (bitmap_later) {
    pack_verdicts_kernel<<<grid_for(ctx, (A.n + 7) / 8, 8), kBlock, 0, st>>>(A.n, A.result, bitmap_later);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return launch_publish(ctx, st, bitmap_later, (A.n + 7) / 8, pw);
  }
  return PBH_OK;
}

// ---- peer windows (include/pbh_b200.h) -----------------------------------------------------------------------------------
static void window_release(pbh_ctx* ctx) {
  for (int r = 0; r < 8; r++) {
    if (ctx->win_peer[r] && ctx->win_peer_ipc[r] && ctx->win_owner) cudaIpcCloseMemHandle(ctx->win_peer[r]);
    ctx->win_peer[r] = nullptr;
    ctx->win_peer_ipc[r] = false;
  }
  if (ctx->win_base && ctx->win_owner) cudaFree(ctx->win_base);
  ctx->win_base = nullptr;
  ctx->win_bytes_per_rank = 0;
  ctx->win_owner = ctx->win_attached = false;
  (void)cudaGetLastError();
}
int pbh_window_create(pbh_ctx* ctx, size_t bytes_per_rank, int rank, int world, void** base_out, uint8_t handle_out[PBH_IPC_HANDLE_BYTES]) {
  CTX_CHECK(ctx);
  static_assert(sizeof(cudaIpcMemHandle_t) == PBH_IPC_HANDLE_BYTES, "IPC handle size");
  if (!base_out || bytes_per_rank == 0 || (bytes_per_rank % 16) != 0 || world < 1 || world > 8 || rank < 0 || rank >= world)
    return fail(ctx, PBH_ERR_BAD_ARGUMENT, "window: 1 <= world <= 8, 0 <= rank < world, bytes_per_rank a positive multiple of 16");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute));
  window_release(ctx);
  CUDA_TRY(ctx, cudaMalloc(&ctx->win_base, bytes_per_rank * (size_t)world));
  CUDA_TRY(ctx, cudaMemset(ctx->win_base, 0, bytes_per_rank * (size_t)world));
  ctx->win_bytes_per_rank = bytes_per_rank;
  ctx->win_rank = rank;
  ctx->win_world = world;
  ctx->win_owner = true;
  if (handle_out) {
    cudaIpcMemHandle_t h;
    CUDA_TRY(ctx, cudaIpcGetMemHandle(&h, ctx->win_base));
    std::memcpy(handle_out, &h, sizeof h);
  }
  *base_out = ctx->win_base;
  return PBH_OK;
}
int pbh_window_attach(pbh_ctx* ctx, const uint8_t* handles) {
  CTX_CHECK(ctx);
  if (!handles || !ctx->win_base || !ctx->win_owner) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "window: create it first");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  for (int r = 0; r < ctx->win_world; r++) {
    if (r == ctx->win_rank) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handles + (size_t)r * PBH_IPC_HANDLE_BYTES, sizeof h);
    void* p = nullptr;
    CUDA_TRY(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->win_peer[r] = static_cast<uint8_t*>(p);
    ctx->win_peer_ipc[r] = true;
  }
  ctx->win_attached = true;
  return PBH_OK;
}
int pbh_window_attach_ptrs(pbh_ctx* ctx, void* const* bases) {
  CTX_CHECK(ctx);
  if (!bases || !ctx->win_base || !ctx->win_owner) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "window: create it first");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  for (int r = 0; r < ctx->win_world; r++) {
    if (r == ctx->win_rank) continue;
    if (!bases[r]) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "window: null peer base");
    cudaPointerAttributes a{};
    CUDA_TRY(ctx, cudaPointerGetAttributes(&a, bases[r]));
    if (a.type != cudaMemoryTypeDevice) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "window: peer base is not device memory");
    if (a.device != ctx->device) {
      int can = 0;
      CUDA_TRY(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, a.device));
      if (!can) return fail(ctx, PBH_ERR_UNSUPPORTED, "window: no peer access to that device");
      cudaError_t e = cudaDeviceEnablePeerAccess(a.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CUDA_TRY(ctx, e);
      (void)cudaGetLastError();
    }
    ctx->win_peer[r] = static_cast<uint8_t*>(bases[r]);
    ctx->win_peer_ipc[r] = false;
  }
  ctx->win_attached = true;
  return PBH_OK;
}
int pbh_window_share(pbh_ctx* owner, pbh_ctx* other) {
  CTX_CHECK(owner);
  CTX_CHECK(other);
  if (owner == other || !owner->win_attached || owner->device != other->device) return fail(owner, PBH_ERR_BAD_ARGUMENT, "window: share an attached window with another context of the same device");
  window_release(other);
  other->win_base = owner->win_base;
  other->win_bytes_per_rank = owner->win_bytes_per_rank;
  other->win_rank = owner->win_rank;
  other->win_world = owner->win_world;
  for (int r = 0; r < 8; r++) other->win_peer[r] = owner->win_peer[r];
  other->win_owner = false;
  other->win_attached = true;
  return PBH_OK;
}
int pbh_window_destroy(pbh_ctx* ctx) {
  CTX_CHECK(ctx);
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = pbh_ctx_sync(ctx);
  window_release(ctx);
  return rc;
}

int pbh_prove_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                        const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !chal || !proof || !status) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || chal_pitch < n || proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ProveArgs A{wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, proof, proof_pitch, status, n};
  return launch_prove(ctx, ctx->compute, A);
}

int pbh_verify_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                         size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !chal || !u || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (proof_pitch < n || chal_pitch < n || (gt && gt_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  VerifyArgs A{proof, proof_pitch, chal, chal_pitch, u, result, gt, gt_pitch, n, nullptr};
  return launch_verify(ctx, ctx->compute, A);
}

int pbh_prove_digest_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                               const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status,
                               uint64_t first_index, uint64_t* digest) {
  CTX_CHECK(ctx);
  if (!digest) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n == 0) { CUDA_TRY(ctx, cudaMemsetAsync(digest, 0, sizeof(uint64_t), ctx->compute)); return PBH_OK; }
  // (no memset otherwise: the fused kernel's last block OVERWRITES *digest with the launch's total, so a captured step is two
  // kernel nodes and nothing else; the unfused path zeroes the word itself)
  if (!wit || !rnd || !chal || !proof || !status) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || chal_pitch < n || proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  ProveArgs A{wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, proof, proof_pitch, status, n};
  return launch_prove(ctx, ctx->compute, A, first_index, digest);
}

int pbh_verify_bitmap_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                                size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* bitmap) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !chal || !u || !result || !bitmap) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (proof_pitch < n || chal_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  VerifyArgs A{proof, proof_pitch, chal, chal_pitch, u, result, nullptr, 0, n, bitmap};
  return launch_verify(ctx, ctx->compute, A);
}

// ---- host-pointer entry points: chunked, double-buffered H2D -> kernel -> D2H ----------------------------
static int ensure_slots(pbh_ctx* ctx, size_t bytes_per_item) {
  size_t need = bytes_per_item * ctx->chunk;
  if (ctx->slot_bytes >= need) return PBH_OK;
  for (int s = 0; s < kSlots; s++) {
    if (ctx->slot_buf[s]) { CUDA_TRY(ctx, cudaFree(ctx->slot_buf[s])); ctx->slot_buf[s] = nullptr; }
    if (ctx->slot_mirror[s]) { CUDA_TRY(ctx, cudaFreeHost(ctx->slot_mirror[s])); ctx->slot_mirror[s] = nullptr; }
  }
  ctx->slot_bytes = 0;
  for (int s = 0; s < kSlots; s++) CUDA_TRY(ctx, cudaMalloc(&ctx->slot_buf[s], need));
  ctx->slot_bytes = need;
  return PBH_OK;
}

// The staged pipeline shared by the host-pointer entry points: the batch is cut into chunks of ctx->chunk items that
// cycle through kSlots staging buffers, each with its own stream, so the upload of chunk k+2, the kernels of chunk k+1
// and the download of chunk k overlap.  `body(lo, m, C, base, stream)` enqueues one chunk of m items starting at item
// lo into the staging buffer `base` (planes of pitch C) on `stream`.
static constexpr size_t kStagePlanes = 128;

// ---- staging rows ----------------------------------------------------------------------------------------------------------
// A body lays its buffers out in rows of C bytes of a staging slot (kStagePlanes rows) or of a lane buffer (the kRows its lane
// call asks for, see lane_call).  Every row range a body uses is named here and nowhere else; the asserts are derived from the names.
struct Rows {
  size_t at, count;
  constexpr size_t end() const { return at + count; }
};
template <class... R>
static constexpr size_t rows_end(R... r) { return std::max({r.end()...}); }
template <class... R>
static constexpr bool rows_disjoint(Rows a, R... r) {   // pairwise
  if constexpr (sizeof...(R) == 0) return true;
  else return ((a.end() <= r.at || r.end() <= a.at) && ...) && rows_disjoint(r...);
}
template <class T = uint8_t>
static T* at_row(uint8_t* base, size_t C, Rows r) { return reinterpret_cast<T*>(base + r.at * C); }

// byte-plane prover, and the verifier fused behind it (pbh_prove_verify_batch, packed_prove_body); also pbh_prove_records
struct ProveRows {
  static constexpr Rows wit{0, 12}, rnd{12, 9}, chal{21, 5}, proof{26, 27}, status{53, 1}, u{54, 1}, res{55, 1};
  static constexpr size_t kRows = rows_end(wit, rnd, chal, proof, status, u, res);
};
// byte-plane verifier (verify_body, packed_verify_body, pbh_verify_records); its proof planes are the prover's rows, where a
// resident packed verify reads what packed_prove_body left
struct VerifyRows {
  static constexpr Rows gt{0, 4}, proof{26, 27}, chal{54, 5}, u{59, 1}, res{60, 1};
  static constexpr size_t kRows = rows_end(gt, proof, chal, u, res);
};
// 32-byte records above the planes (pbh_prove_records, pbh_verify_records)
struct RecordRows {
  static constexpr Rows witness{64, 32}, proof{96, 32};
};
// packed records above the planes: prover input and output, verifier input (packed proofs, challenge words)
struct PackedRows {
  static constexpr Rows in{64, sizeof(pbh_packed_witness)}, out{80, sizeof(pbh_packed_proof)};
  static constexpr Rows proofs{96, sizeof(pbh_packed_proof)}, chal_u{108, sizeof(uint32_t)};
  static constexpr size_t kProveRows = std::max(ProveRows::kRows, rows_end(in, out)), kVerifyRows = std::max(VerifyRows::kRows, rows_end(proofs, chal_u));
};
// Fiat-Shamir byte planes (pbh_prove_fs_batch, pbh_verify_fs_batch): the prover's or the verifier's rows, and the challenges out
struct FsRows {
  static constexpr Rows chal_out{54, 6};
};
// Fiat-Shamir packed records: the prover's records, proofs and challenge words; the verifier's proofs and results
struct FsPackedRows {
  static constexpr Rows in{64, sizeof(pbh_packed_fs_witness)}, out{80, sizeof(pbh_packed_proof)}, chal_u{92, sizeof(uint32_t)};
  static constexpr Rows proofs{96, sizeof(pbh_packed_proof)}, res{108, 1};
  static constexpr size_t kProveRows = rows_end(in, out, chal_u), kVerifyRows = rows_end(proofs, res);
};
using PR = ProveRows;
using VR = VerifyRows;
static_assert(rows_disjoint(PR::wit, PR::rnd, PR::chal, PR::proof, PR::status, PR::u, PR::res) && rows_disjoint(VR::gt, VR::proof, VR::chal, VR::u, VR::res) &&
                  rows_disjoint(PR::wit, PR::rnd, PR::proof, PR::status, FsRows::chal_out) && rows_disjoint(VR::gt, VR::proof, VR::res, FsRows::chal_out) &&
                  rows_disjoint(RecordRows::witness, RecordRows::proof) &&
                  std::max({PR::kRows, VR::kRows, FsRows::chal_out.end()}) <= std::min(RecordRows::witness.at, PackedRows::in.at),
              "no body uses a row twice; records sit above the planes");
static_assert(std::max({PackedRows::kProveRows, PackedRows::kVerifyRows, RecordRows::proof.end(), FsPackedRows::kProveRows, FsPackedRows::kVerifyRows,
}) <= kStagePlanes,
              "every body fits a staging slot");
static_assert(rows_disjoint(PackedRows::in, PackedRows::out, PackedRows::proofs, PackedRows::chal_u) &&
                  rows_disjoint(FsPackedRows::in, FsPackedRows::out, FsPackedRows::chal_u, FsPackedRows::proofs, FsPackedRows::res),
              "the prover's and the verifier's packed records are disjoint");
static_assert(VR::proof.at == PR::proof.at && VR::proof.count == PR::proof.count && rows_disjoint(PR::proof, VR::chal, VR::u, VR::res, PackedRows::chal_u),
              "resident proofs: packed_verify_body reads the proof planes packed_prove_body left and writes none of them");
static bool host_pinned(const void* p);
static int slot_of(const pbh_ctx* ctx, const uint8_t* base) {
  for (int s = 0; s < kSlots; s++)
    if (ctx->slot_buf[s] && ctx->slot_buf[s] == base) return s;
  return -1;
}
// the page-locked mirror of slot s (and the thread pool), created on first use
static int ensure_mirror(pbh_ctx* ctx, int s) {
  if (!ctx->slot_mirror[s]) CUDA_TRY(ctx, cudaHostAlloc(&ctx->slot_mirror[s], ctx->slot_bytes, cudaHostAllocDefault));
  if (!ctx->pool) {
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    ctx->pool = new CopyPool((int)std::min(6u, std::max(1u, hw / 4)));
  }
  return PBH_OK;
}
static void row_tasks(std::vector<CopyTask>& out, uint8_t* dst, size_t dpitch, const uint8_t* src, size_t spitch, size_t width, size_t rows) {
  constexpr size_t kSeg = (size_t)256 << 10;   // a row is cut into 256 KiB segments so that a single long row also spreads over the pool
  for (size_t r = 0; r < rows; r++)
    for (size_t o = 0; o < width; o += kSeg) out.push_back({dst + r * dpitch + o, src + r * spitch + o, std::min(kSeg, width - o)});
}
// `rows` rows of `width` bytes from caller memory (pitch hpitch) into the staging buffer `base` at dev (pitch dpitch), on st
static int stage_h2d(pbh_ctx* ctx, uint8_t* base, cudaStream_t st, void* dev_, size_t dpitch, const void* host_, size_t hpitch, size_t width,
                     size_t rows) {
  uint8_t* dev = static_cast<uint8_t*>(dev_);
  const uint8_t* host = static_cast<const uint8_t*>(host_);
  if (rows == 1) dpitch = hpitch = width;
  const int s = ctx->host_stage ? slot_of(ctx, base) : -1;
  if (s < 0 || host_pinned(host)) {
    CUDA_TRY(ctx, cudaMemcpy2DAsync(dev, dpitch, host, hpitch, width, rows, cudaMemcpyHostToDevice, st));
    return PBH_OK;
  }
  PBH_TRY(ensure_mirror(ctx, s));
  uint8_t* mir = ctx->slot_mirror[s] + (dev - base);
  std::vector<CopyTask> tasks;
  row_tasks(tasks, mir, dpitch, host, hpitch, width, rows);
  ctx->pool->run(tasks);
  ctx->slot_dirty[s] = true;
  CUDA_TRY(ctx, cudaMemcpy2DAsync(dev, dpitch, mir, dpitch, width, rows, cudaMemcpyHostToDevice, st));
  return PBH_OK;
}
// the reverse: results at dev go to caller memory, directly (page-locked) or through the mirror (copied out by flush_slot)
static int stage_d2h(pbh_ctx* ctx, uint8_t* base, cudaStream_t st, void* host_, size_t hpitch, const void* dev_, size_t dpitch, size_t width,
                     size_t rows) {
  const uint8_t* dev = static_cast<const uint8_t*>(dev_);
  uint8_t* host = static_cast<uint8_t*>(host_);
  if (rows == 1) dpitch = hpitch = width;
  const int s = ctx->host_stage ? slot_of(ctx, base) : -1;
  if (s < 0 || host_pinned(host)) {
    CUDA_TRY(ctx, cudaMemcpy2DAsync(host, hpitch, dev, dpitch, width, rows, cudaMemcpyDeviceToHost, st));
    return PBH_OK;
  }
  PBH_TRY(ensure_mirror(ctx, s));
  uint8_t* mir = ctx->slot_mirror[s] + (dev - base);
  CUDA_TRY(ctx, cudaMemcpy2DAsync(mir, dpitch, dev, dpitch, width, rows, cudaMemcpyDeviceToHost, st));
  row_tasks(ctx->slot_out[s], host, hpitch, mir, dpitch, width, rows);
  ctx->slot_dirty[s] = true;
  return PBH_OK;
}
// waits for slot s and delivers the outputs parked in its mirror
static int flush_slot(pbh_ctx* ctx, int s) {
  if (!ctx->slot_dirty[s]) return PBH_OK;
  cudaError_t e = cudaStreamSynchronize(ctx->slot_stream[s]);
  ctx->slot_dirty[s] = false;
  if (e != cudaSuccess) {
    ctx->slot_out[s].clear();
    ctx->last_error = std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e);
    return PBH_ERR_CUDA;
  }
  if (!ctx->slot_out[s].empty()) ctx->pool->run(ctx->slot_out[s]);
  ctx->slot_out[s].clear();
  return PBH_OK;
}
template <class Body>
static int for_each_chunk(pbh_ctx* ctx, size_t n, Body body, bool wait = true) {
  // a synchronous call starts after everything the lanes (which share these streams) were given: it may read a buffer an
  // asynchronous call is still filling
  for (int s = 0; s < kSlots; s++) {
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot_stream[s]));
    ctx->resident_host[s] = nullptr;
  }
  int rc = ensure_slots(ctx, kStagePlanes);
  if (rc) return rc;
  const size_t C = ctx->chunk;
  size_t k = 0;
  for (size_t lo = 0; lo < n && rc == PBH_OK; lo += C, k++) {
    const int s = (int)(k % kSlots);
    rc = flush_slot(ctx, s);          // the slot's mirror is about to be overwritten
    if (rc == PBH_OK) rc = body(lo, std::min(C, n - lo), C, ctx->slot_buf[s], ctx->slot_stream[s]);
  }
  for (int s = 0; s < kSlots; s++) {
    if (rc == PBH_OK) rc = flush_slot(ctx, s);
    else { ctx->slot_out[s].clear(); }
  }
  // Also on failure: copies that read or write the caller's buffers may still be in flight, and the caller is free to
  // release them as soon as this call returns.
  if (rc != PBH_OK || wait) {
    const std::string keep = ctx->last_error;
    for (int s = 0; s < kSlots; s++) {
      cudaError_t e = cudaStreamSynchronize(ctx->slot_stream[s]);
      if (e != cudaSuccess && rc == PBH_OK) { ctx->last_error = std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e); rc = PBH_ERR_CUDA; }
    }
    if (rc != PBH_OK && !keep.empty() && ctx->last_error.empty()) ctx->last_error = keep;
  }
  return rc;
}

// The device-side alias of a host range when the whole range is page-locked and mapped (cudaHostAlloc /
// cudaHostRegister under unified addressing), else nullptr.  When every buffer of a host-pointer call has one, the tile
// kernel runs in place on the caller's memory: its TMA loads and stores cross PCIe tile by tile, so upload, compute and
// download overlap at 256-item granularity with no staging copy, no pipeline fill/drain and one launch.  Measured on
// PCIe Gen5 x16 (scripts/time_zero_copy.py): prove 0.83 ms per 2^20 items against 0.97 ms for the best staged chunking
// (the copy engine pays about a microsecond per row of a pitched copy, which bounds how small a staged chunk can be).
typedef CUresult (*PointerGetAttributeFn)(void*, CUpointer_attribute, CUdeviceptr);
static PointerGetAttributeFn pointer_get_attribute_fn() {
  static PointerGetAttributeFn fn = []() -> PointerGetAttributeFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuPointerGetAttribute", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      return nullptr;
    return (PointerGetAttributeFn)p;
  }();
  return fn;
}
// The whole span [p, p + span) must lie inside ONE page-locked, mapped allocation or registration: the range the driver
// reports for the first byte has to cover the last one too (probing the two ends alone would accept two registrations
// with an unmapped hole between them, and the kernel would fault on the hole).  Anything else takes the staged path.
static uint8_t* mapped_host_alias(pbh_ctx* ctx, const uint8_t* p, size_t span) {
  if (!ctx->host_direct || !p || span == 0) return nullptr;
  cudaPointerAttributes lo{};
  if (cudaPointerGetAttributes(&lo, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (lo.type != cudaMemoryTypeHost || !lo.devicePointer) return nullptr;
  PointerGetAttributeFn attr = pointer_get_attribute_fn();
  if (!attr) return nullptr;
  CUdeviceptr start = 0;
  size_t size = 0;
  if (attr(&start, CU_POINTER_ATTRIBUTE_RANGE_START_ADDR, (CUdeviceptr)(uintptr_t)lo.devicePointer) != CUDA_SUCCESS ||
      attr(&size, CU_POINTER_ATTRIBUTE_RANGE_SIZE, (CUdeviceptr)(uintptr_t)lo.devicePointer) != CUDA_SUCCESS)
    return nullptr;
  const uintptr_t a = (uintptr_t)lo.devicePointer;
  if (a < (uintptr_t)start || a + span > (uintptr_t)start + size) return nullptr;
  return (uint8_t*)lo.devicePointer;
}

// One byte-plane prove of A.n items on st.  Each direction either goes through rows of `base` by the copy engines (A holds the
// caller's host buffers for it) or is read / written by the kernel in place (A holds device or mapped memory for it).
static int prove_body(pbh_ctx* ctx, cudaStream_t st, uint8_t* base, size_t C, ProveArgs A, bool stage_in, bool stage_out) {
  const ProveArgs H = A;
  if (stage_in) {
    uint8_t *wit = at_row(base, C, PR::wit), *rnd = at_row(base, C, PR::rnd), *chal = at_row(base, C, PR::chal);
    PBH_TRY(stage_h2d(ctx, base, st, wit, C, H.wit, H.wit_pitch, A.n, PR::wit.count));
    PBH_TRY(stage_h2d(ctx, base, st, rnd, C, H.rnd, H.rand_pitch, A.n, PR::rnd.count));
    PBH_TRY(stage_h2d(ctx, base, st, chal, C, H.chal, H.chal_pitch, A.n, PR::chal.count));
    A.wit = wit; A.rnd = rnd; A.chal = chal;
    A.wit_pitch = A.rand_pitch = A.chal_pitch = C;
  }
  if (stage_out) { A.proof = at_row(base, C, PR::proof); A.proof_pitch = C; A.status = at_row(base, C, PR::status); }
  PBH_TRY(launch_prove(ctx, st, A));
  if (stage_out) {
    PBH_TRY(stage_d2h(ctx, base, st, H.proof, H.proof_pitch, A.proof, C, A.n, PR::proof.count));
    PBH_TRY(stage_d2h(ctx, base, st, H.status, 0, A.status, 0, A.n, 1));
  }
  return PBH_OK;
}
// One byte-plane verify, with the same choice per direction.
static int verify_body(pbh_ctx* ctx, cudaStream_t st, uint8_t* base, size_t C, VerifyArgs A, bool stage_in, bool stage_out) {
  const VerifyArgs H = A;
  if (stage_in) {
    uint8_t *proof = at_row(base, C, VR::proof), *chal = at_row(base, C, VR::chal), *u = at_row(base, C, VR::u);
    PBH_TRY(stage_h2d(ctx, base, st, proof, C, H.proof, H.proof_pitch, A.n, VR::proof.count));
    PBH_TRY(stage_h2d(ctx, base, st, chal, C, H.chal, H.chal_pitch, A.n, VR::chal.count));
    PBH_TRY(stage_h2d(ctx, base, st, u, 0, H.u, 0, A.n, 1));
    A.proof = proof; A.chal = chal; A.u = u;
    A.proof_pitch = A.chal_pitch = C;
  }
  if (stage_out) {
    A.result = at_row(base, C, VR::res);
    if (A.gt) { A.gt = at_row(base, C, VR::gt); A.gt_pitch = C; }
  }
  PBH_TRY(launch_verify(ctx, st, A));
  if (stage_out) {
    PBH_TRY(stage_d2h(ctx, base, st, H.result, 0, A.result, 0, A.n, 1));
    if (H.gt) PBH_TRY(stage_d2h(ctx, base, st, H.gt, H.gt_pitch, A.gt, C, A.n, VR::gt.count));
  }
  return PBH_OK;
}
// The buffers of A replaced by their mapped device aliases (nullptr where there is none; a null gt stays null)
static ProveArgs mapped(pbh_ctx* ctx, const ProveArgs& A) {
  return ProveArgs{mapped_host_alias(ctx, A.wit, 11 * A.wit_pitch + A.n), A.wit_pitch, mapped_host_alias(ctx, A.rnd, 8 * A.rand_pitch + A.n),
                   A.rand_pitch, mapped_host_alias(ctx, A.chal, 4 * A.chal_pitch + A.n), A.chal_pitch,
                   mapped_host_alias(ctx, A.proof, 26 * A.proof_pitch + A.n), A.proof_pitch, mapped_host_alias(ctx, A.status, A.n), A.n};
}
static VerifyArgs mapped(pbh_ctx* ctx, const VerifyArgs& A) {
  return VerifyArgs{mapped_host_alias(ctx, A.proof, 26 * A.proof_pitch + A.n), A.proof_pitch, mapped_host_alias(ctx, A.chal, 4 * A.chal_pitch + A.n),
                    A.chal_pitch, mapped_host_alias(ctx, A.u, A.n), mapped_host_alias(ctx, A.result, A.n),
                    A.gt ? mapped_host_alias(ctx, A.gt, 3 * A.gt_pitch + A.n) : nullptr, A.gt_pitch, A.n, nullptr};
}

int pbh_prove_batch(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                    const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !chal || !proof || !status) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || chal_pitch < n || proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const ProveArgs M = mapped(ctx, ProveArgs{wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, proof, proof_pitch, status, n});
  if (M.wit && M.rnd && M.chal && M.proof && M.status) {   // everything mapped: the body in place, one launch
    PBH_TRY(launch_prove(ctx, ctx->slot_stream[0], M));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    return PBH_OK;
  }
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    const ProveArgs A{wit + lo, wit_pitch, rnd + lo, rand_pitch, chal + lo, chal_pitch, proof + lo, proof_pitch, status + lo, m};
    return prove_body(ctx, st, base, C, A, true, true);
  });
}

int pbh_verify_batch(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal, size_t chal_pitch,
                     const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !chal || !u || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (proof_pitch < n || chal_pitch < n || (gt && gt_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const VerifyArgs M = mapped(ctx, VerifyArgs{proof, proof_pitch, chal, chal_pitch, u, result, gt, gt_pitch, n, nullptr});
  if (M.proof && M.chal && M.u && M.result && (!gt || M.gt)) {
    PBH_TRY(launch_verify(ctx, ctx->slot_stream[0], M));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot_stream[0]));
    return PBH_OK;
  }
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    const VerifyArgs A{proof + lo, proof_pitch, chal + lo, chal_pitch, u + lo, result + lo, gt ? gt + lo : nullptr, gt_pitch, m, nullptr};
    return verify_body(ctx, st, base, C, A, true, true);
  });
}

// prove then verify without the proof leaving the device in between: per chunk, H2D inputs -> prove kernel -> verify
// kernel -> D2H proof + status + result
int pbh_prove_verify_batch(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                           const uint8_t* chal, size_t chal_pitch, const uint8_t* u, uint8_t* proof, size_t proof_pitch,
                           uint8_t* status, uint8_t* result) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !chal || !u || !proof || !status || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || chal_pitch < n || proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    uint8_t *d_wit = at_row(base, C, PR::wit), *d_rnd = at_row(base, C, PR::rnd), *d_chal = at_row(base, C, PR::chal),
            *d_proof = at_row(base, C, PR::proof), *d_status = at_row(base, C, PR::status), *d_u = at_row(base, C, PR::u),
            *d_res = at_row(base, C, PR::res);
    PBH_TRY(stage_h2d(ctx, base, st, d_wit, C, wit + lo, wit_pitch, m, PR::wit.count));
    PBH_TRY(stage_h2d(ctx, base, st, d_rnd, C, rnd + lo, rand_pitch, m, PR::rnd.count));
    PBH_TRY(stage_h2d(ctx, base, st, d_chal, C, chal + lo, chal_pitch, m, PR::chal.count));
    PBH_TRY(stage_h2d(ctx, base, st, d_u, 0, u + lo, 0, m, 1));
    ProveArgs A{d_wit, C, d_rnd, C, d_chal, C, d_proof, C, d_status, m};
    int rc = launch_prove(ctx, st, A);
    if (rc) return rc;
    VerifyArgs V{d_proof, C, d_chal, C, d_u, d_res, nullptr, 0, m, nullptr};
    rc = launch_verify(ctx, st, V);
    if (rc) return rc;
    PBH_TRY(stage_d2h(ctx, base, st, proof + lo, proof_pitch, d_proof, C, m, PR::proof.count));
    PBH_TRY(stage_d2h(ctx, base, st, status + lo, 0, d_status, 0, m, 1));
    PBH_TRY(stage_d2h(ctx, base, st, result + lo, 0, d_res, 0, m, 1));
    return PBH_OK;
  });
}

// ---- asynchronous host-pointer calls (include/pbh_b200.h "lanes") ------------------------------------------------------
// A lane is one of the context's slot streams, with a whole-batch staging buffer.  Page-locked buffers travel on the lane's
// stream and the call returns at once.  Kernels that read or write mapped host memory in place run on half grids (one prover
// block and two verifier blocks per SM), so that kernels of different lanes are resident together and the upload of one batch
// shares the link with the download of another.  Other buffers take the synchronous staged path (copies from pageable memory
// are synchronous anyway).  Calls on one lane run in issue order, so a call may reuse the rows of the lane buffer the previous
// one used; the proof planes a packed prove leaves there are the one thing a later call (a resident verify) reads.
static int lane_stream(pbh_ctx* ctx, int lane, cudaStream_t* st) {
  if (lane < 0 || lane >= PBH_LANES) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "lane out of range");
  *st = ctx->slot_stream[lane];
  return PBH_OK;
}
// page-locked (mapped or not): the copy engines can read and write it asynchronously
static bool host_pinned(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}
// whole-batch staging buffer of a lane: `rows` planes of pitch C = n rounded up to a tile
static int ensure_lane(pbh_ctx* ctx, int lane, size_t bytes) {
  if (ctx->lane_bytes[lane] >= bytes) return PBH_OK;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot_stream[lane]));
  if (ctx->lane_buf[lane]) { CUDA_TRY(ctx, cudaFree(ctx->lane_buf[lane])); ctx->lane_buf[lane] = nullptr; ctx->lane_bytes[lane] = 0; }
  CUDA_TRY(ctx, cudaMalloc(&ctx->lane_buf[lane], bytes));
  ctx->lane_bytes[lane] = bytes;
  return PBH_OK;
}
static constexpr size_t kLaneMaxItems = (size_t)1 << 24;   // larger batches take the synchronous chunked path

// How a lane call's buffers travel
struct LanePlan {
  bool async;      // on the lane; else the call waits for the context and runs synchronously
  size_t rows;     // lane-buffer rows the body stages through (0: none)
  bool in_place;   // a kernel reads or writes mapped host memory (half grids)
};
// every buffer (null ones aside) page-locked and the batch within kLaneMaxItems: all of it through the lane buffer
static LanePlan staged_plan(size_t n, size_t rows, std::initializer_list<const void*> bufs) {
  bool ok = n <= kLaneMaxItems;
  for (const void* p : bufs) ok = ok && (!p || host_pinned(p));
  return {ok, rows, false};
}
// a byte-plane call (PBH_OPT_LANE_MODE): each direction through the lane buffer by the copy engine (its mode bit set, or
// page-locked memory that is not mapped) or in place on mapped memory
static LanePlan plane_plan(const pbh_ctx* ctx, size_t n, size_t rows, bool in_pinned, bool in_mapped, bool out_pinned, bool out_mapped,
                           bool* stage_in, bool* stage_out) {
  *stage_in = in_pinned && ((ctx->lane_mode & 1) || !in_mapped) && n <= kLaneMaxItems;
  *stage_out = out_pinned && ((ctx->lane_mode & 2) || !out_mapped) && n <= kLaneMaxItems;
  return {(*stage_in || in_mapped) && (*stage_out || out_mapped), (*stage_in || *stage_out) ? rows : 0, !(*stage_in && *stage_out)};
}

// Every lane call (include/pbh_b200.h "lanes"): the lane is checked and its resident proofs are forgotten; n == 0 returns; `bad`
// is what is wrong with the caller's arguments, or nullptr.  `plan()` then decides: buffers that cannot travel on the lane take
// the synchronous call `sync()` once everything enqueued on the context is done (it shares the slot streams with the lanes).
// Otherwise the lane buffer is grown to plan.rows rows of C = n rounded up to a tile and `body(stream, lane buffer, C, resident)`
// enqueues the batch; `resident` is the host buffer whose proofs the previous call on the lane left in the lane buffer, when
// it had this n and the buffer was not reallocated since.  A body that fails may already have enqueued copies of the caller's
// buffers: the call waits for the lane before it returns the error, since the caller may release them once it has returned.
template <class Plan, class Body, class Sync>
static int lane_call(pbh_ctx* ctx, int lane, size_t n, const char* bad, Plan plan, Body body, Sync sync) {
  cudaStream_t st;
  PBH_TRY(lane_stream(ctx, lane, &st));
  const void* resident = ctx->resident_n[lane] == n ? ctx->resident_host[lane] : nullptr;
  ctx->resident_host[lane] = nullptr;
  if (n == 0) return PBH_OK;
  if (bad) return fail(ctx, PBH_ERR_BAD_ARGUMENT, bad);
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const LanePlan p = plan();
  if (!p.async) {
    PBH_TRY(pbh_ctx_sync(ctx));
    return sync();
  }
  const size_t C = (n + kTile - 1) / kTile * kTile;
  if (p.rows) {
    const size_t had = ctx->lane_bytes[lane];
    PBH_TRY(ensure_lane(ctx, lane, p.rows * C));
    if (ctx->lane_bytes[lane] != had) resident = nullptr;
  }
  const int keep = ctx->grid_scale;
  if (p.in_place) ctx->grid_scale = 1;
  const int rc = body(st, ctx->lane_buf[lane], C, resident);
  ctx->grid_scale = keep;
  if (rc != PBH_OK) {
    const std::string err = ctx->last_error;
    cudaStreamSynchronize(st);
    cudaGetLastError();
    ctx->last_error = err;
  }
  return rc;
}

int pbh_prove_batch_async(pbh_ctx* ctx, int lane, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                          const uint8_t* chal, size_t chal_pitch, uint8_t* proof, size_t proof_pitch, uint8_t* status) {
  CTX_CHECK(ctx);
  const char* bad = !wit || !rnd || !chal || !proof || !status ? "null pointer"
                    : wit_pitch < n || rand_pitch < n || chal_pitch < n || proof_pitch < n ? "pitch < n" : nullptr;
  ProveArgs A{wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, proof, proof_pitch, status, n};
  bool stage_in = false, stage_out = false;
  return lane_call(ctx, lane, n, bad,
      [&] {
        const ProveArgs M = mapped(ctx, A);
        const LanePlan p = plane_plan(ctx, n, PR::kRows, host_pinned(wit) && host_pinned(rnd) && host_pinned(chal), M.wit && M.rnd && M.chal,
                                      host_pinned(proof) && host_pinned(status), M.proof && M.status, &stage_in, &stage_out);
        if (!stage_in) { A.wit = M.wit; A.rnd = M.rnd; A.chal = M.chal; }
        if (!stage_out) { A.proof = M.proof; A.status = M.status; }
        return p;
      },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void*) { return prove_body(ctx, st, base, C, A, stage_in, stage_out); },
      [&] { return pbh_prove_batch(ctx, n, wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, proof, proof_pitch, status); });
}
int pbh_verify_batch_async(pbh_ctx* ctx, int lane, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* chal,
                           size_t chal_pitch, const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch) {
  CTX_CHECK(ctx);
  const char* bad = !proof || !chal || !u || !result ? "null pointer"
                    : proof_pitch < n || chal_pitch < n || (gt && gt_pitch < n) ? "pitch < n" : nullptr;
  VerifyArgs A{proof, proof_pitch, chal, chal_pitch, u, result, gt, gt_pitch, n, nullptr};
  bool stage_in = false, stage_out = false;
  return lane_call(ctx, lane, n, bad,
      [&] {
        const VerifyArgs M = mapped(ctx, A);
        const LanePlan p = plane_plan(ctx, n, VR::kRows, host_pinned(proof) && host_pinned(chal) && host_pinned(u), M.proof && M.chal && M.u,
                                      host_pinned(result) && (!gt || host_pinned(gt)), M.result && (!gt || M.gt), &stage_in, &stage_out);
        if (!stage_in) { A.proof = M.proof; A.chal = M.chal; A.u = M.u; }
        if (!stage_out) { A.result = M.result; A.gt = M.gt; }
        return p;
      },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void*) { return verify_body(ctx, st, base, C, A, stage_in, stage_out); },
      [&] { return pbh_verify_batch(ctx, n, proof, proof_pitch, chal, chal_pitch, u, result, gt, gt_pitch); });
}
int pbh_lane_sync(pbh_ctx* ctx, int lane) {
  CTX_CHECK(ctx);
  cudaStream_t st;
  PBH_TRY(lane_stream(ctx, lane, &st));
  ctx->resident_host[lane] = nullptr;   // after a sync the caller may change its buffers
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return PBH_OK;
}

// ---- page-locked, mapped host memory next to the device ------------------------------------------------------------------
// NUMA node of the device's PCIe root from sysfs (-1: the platform, e.g. a virtual machine, does not expose one)
static int device_numa_node(int device) {
  char id[32] = {0};
  if (cudaDeviceGetPCIBusId(id, sizeof id, device) != cudaSuccess) { cudaGetLastError(); return -1; }
  for (char* c = id; *c; c++) *c = (char)std::tolower((unsigned char)*c);
  std::string path = std::string("/sys/bus/pci/devices/") + id + "/numa_node";
  FILE* f = std::fopen(path.c_str(), "r");
  if (!f) return -1;
  int node = -1;
  if (std::fscanf(f, "%d", &node) != 1) node = -1;
  std::fclose(f);
  return node;
}
int pbh_ctx_numa_node(const pbh_ctx* ctx) { return ctx ? ctx->numa_node : PBH_ERR_BAD_ARGUMENT; }

int pbh_host_alloc(pbh_ctx* ctx, size_t bytes, void** out) {
  CTX_CHECK(ctx);
  if (!out || bytes == 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer or zero size");
  *out = nullptr;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (ctx->numa_node >= 0 && ctx->numa_node < 1024) {
    // pages bound to the device's node (mbind, MPOL_BIND = 2), touched, then page-locked and mapped
    const size_t page = (size_t)sysconf(_SC_PAGESIZE), len = (bytes + page - 1) / page * page;
    void* p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p != MAP_FAILED) {
      unsigned long mask[16] = {0};
      mask[ctx->numa_node / (8 * sizeof(unsigned long))] |= 1ul << (ctx->numa_node % (8 * sizeof(unsigned long)));
      const long mb = syscall(SYS_mbind, p, len, 2 /* MPOL_BIND */, mask, (unsigned long)(8 * sizeof mask), 0u);
      if (mb == 0) {
        for (size_t o = 0; o < len; o += page) static_cast<volatile uint8_t*>(p)[o] = 0;
        if (cudaHostRegister(p, len, cudaHostRegisterPortable | cudaHostRegisterMapped) == cudaSuccess) {
          ctx->host_allocs[p] = {len, true};
          *out = p;
          return PBH_OK;
        }
        cudaGetLastError();
      }
      munmap(p, len);
    }
  }
  void* p = nullptr;
  CUDA_TRY(ctx, cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocMapped));
  ctx->host_allocs[p] = {bytes, false};
  *out = p;
  return PBH_OK;
}
// Page-locked WRITE-COMBINED memory for buffers the host only writes and the device only reads (inputs): the device's reads
// of it need no snoop of the CPU caches.  CPU reads of such memory are uncached and very slow - never use it for outputs.
int pbh_host_alloc_input(pbh_ctx* ctx, size_t bytes, void** out) {
  CTX_CHECK(ctx);
  if (!out || bytes == 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer or zero size");
  *out = nullptr;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  void* p = nullptr;
  CUDA_TRY(ctx, cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocMapped | cudaHostAllocWriteCombined));
  ctx->host_allocs[p] = {bytes, false};
  *out = p;
  return PBH_OK;
}
int pbh_host_free(pbh_ctx* ctx, void* p) {
  CTX_CHECK(ctx);
  if (!p) return PBH_OK;
  auto it = ctx->host_allocs.find(p);
  if (it == ctx->host_allocs.end()) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "not a pbh_host_alloc pointer of this context");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = pbh_ctx_sync(ctx);
  if (it->second.second) { cudaHostUnregister(p); munmap(p, it->second.first); } else cudaFreeHost(p);
  ctx->host_allocs.erase(it);
  return rc;
}

// ---- Fiat-Shamir entry points (SURVEY.md §8(f) row 1) -----------------------------------------------------------------
static FsSeed fs_seed_of(const pbh_ctx* ctx) {
  FsSeed s;
  for (int i = 0; i < 8; i++) s.w[i] = ctx->hs.fs_seed[i];
  return s;
}
int pbh_ctx_get_fs_seed(const pbh_ctx* ctx, uint8_t seed[32]) {
  if (!ctx || !seed) return PBH_ERR_BAD_ARGUMENT;
  for (int i = 0; i < 8; i++)
    for (int b = 0; b < 4; b++) seed[4 * i + b] = (uint8_t)(ctx->hs.fs_seed[i] >> (24 - 8 * b));
  return PBH_OK;
}
// The compile-time <ALGO, FP32, PBH_CIRCUIT> of the Fiat-Shamir provers for a context, handed to f as an FsProver<...>.  Five
// instantiations: both algorithms with the FP32 or the int32 prover, and the TABLE FP32 prover for the reference's own circuit.
template <int ALGO, bool FP32, bool PBH_CIRCUIT>
struct FsProver {
  static constexpr int algo = ALGO;
  static constexpr bool fp32 = FP32, pbh_circuit = PBH_CIRCUIT;
};
template <class F>
static void with_fs_prover(const pbh_ctx* ctx, F f) {
  const bool special = ctx->pbh_circuit && ctx->specialise;
  if (ctx->algo == PBH_ALGO_TABLE) {
    if (!ctx->prover_fp32) f(FsProver<ALGO_TABLE, false, false>{});
    else if (special) f(FsProver<ALGO_TABLE, true, true>{});
    else f(FsProver<ALGO_TABLE, true, false>{});
  } else {
    if (!ctx->prover_fp32) f(FsProver<ALGO_ARITH, false, false>{});
    else f(FsProver<ALGO_ARITH, true, false>{});
  }
}
// The same for the Fiat-Shamir verifiers: <ALGO> as a std::integral_constant, and the run-time fp32 flag (TABLE only).
template <class F>
static void with_fs_verifier(const pbh_ctx* ctx, F f) {
  if (ctx->algo == PBH_ALGO_TABLE) f(std::integral_constant<int, ALGO_TABLE>{}, ctx->verifier_fp32 != 0);
  else f(std::integral_constant<int, ALGO_ARITH>{}, false);
}

// digest (nullable): device uint64, overwritten with the digest of the 27 proof planes (items first_index ..).  The FP32 provers
// add it in the kernel (launch-local record, no memset); the int32 prover has no such instantiation and runs the digest kernel
// on a zeroed word after it, as launch_prove does off the TMA path.
static int launch_prove_fs(pbh_ctx* ctx, cudaStream_t st, const ProveFsArgs& F, uint64_t first_index = 0, uint64_t* digest = nullptr) {
  if (F.base.n == 0) return PBH_OK;
  const int grid = grid_for(ctx, F.base.n, 2);
  const FsSeed seed = fs_seed_of(ctx);
  const bool fused = digest && ctx->prover_fp32;
  FsDigestArgs D{};
  if (fused) {
    unsigned int* tc = fresh_tile_counter(ctx, st);
    if (!tc) return fail(ctx, PBH_ERR_UNSUPPORTED, "too many launches captured into CUDA graphs from this context");
    D = FsDigestArgs{first_index, (unsigned long long*)digest, tc, peer_window_for(ctx, digest, sizeof(uint64_t))};
  }
  with_fs_prover(ctx, [&](auto P) {
    using I = decltype(P);
    if constexpr (I::fp32) {
      if (fused) {
        prove_fs_kernel<I::algo, true, I::pbh_circuit, true><<<grid, 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, seed, ctx->d_tables, F, D);
        return;
      }
    }
    prove_fs_kernel<I::algo, I::fp32, I::pbh_circuit><<<grid, 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, seed, ctx->d_tables, F, D);
  });
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  if (digest && !fused) {
    CUDA_TRY(ctx, cudaMemsetAsync(digest, 0, sizeof(uint64_t), st));
    PBH_TRY(launch_digest(ctx, st, F.base.n, first_index, 27, F.base.proof, F.base.proof_pitch, digest));
    return launch_publish(ctx, st, digest, sizeof(uint64_t), peer_window_for(ctx, digest, sizeof(uint64_t)));
  }
  return PBH_OK;
}
// F.base.bitmap (nullable): the verdict bitmap, packed in the kernel when it is 4-byte aligned, by pack_verdicts_kernel after it
// otherwise (as launch_verify does); with a peer window it is also stored into every peer's.
static int launch_verify_fs(pbh_ctx* ctx, cudaStream_t st, const VerifyFsArgs& F) {
  if (F.base.n == 0) return PBH_OK;
  const int grid = grid_for(ctx, F.base.n, 2);
  const FsSeed seed = fs_seed_of(ctx);
  uint8_t* bitmap = F.base.bitmap;
  const PeerWindow pw = peer_window_for(ctx, bitmap, (F.base.n + 7) / 8);
  const bool fused = bitmap && ((uintptr_t)bitmap % 4) == 0;
  with_fs_verifier(ctx, [&](auto algo, bool fp32) {
    if (fused) verify_fs_kernel<decltype(algo)::value, true><<<grid, 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, fp32, seed, ctx->d_tables, F, pw);
    else verify_fs_kernel<decltype(algo)::value><<<grid, 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, fp32, seed, ctx->d_tables, F, PeerWindow{});
  });
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  if (bitmap && !fused) {
    pack_verdicts_kernel<<<grid_for(ctx, (F.base.n + 7) / 8, 8), kBlock, 0, st>>>(F.base.n, F.base.result, bitmap);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return launch_publish(ctx, st, bitmap, (F.base.n + 7) / 8, pw);
  }
  return PBH_OK;
}

int pbh_prove_fs_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                           uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !proof || !status) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || proof_pitch < n || (chal_out && chal_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ProveFsArgs F{{wit, wit_pitch, rnd, rand_pitch, nullptr, 0, proof, proof_pitch, status, n}, chal_out, chal_pitch};
  return launch_prove_fs(ctx, ctx->compute, F);
}
int pbh_verify_fs_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result, uint8_t* chal_out,
                            size_t chal_pitch, uint8_t* gt, size_t gt_pitch) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (proof_pitch < n || (chal_out && chal_pitch < n) || (gt && gt_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  VerifyFsArgs F{{proof, proof_pitch, nullptr, 0, nullptr, result, gt, gt_pitch, n, nullptr}, chal_out, chal_pitch};
  return launch_verify_fs(ctx, ctx->compute, F);
}
int pbh_prove_fs_digest_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                                  uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch,
                                  uint64_t first_index, uint64_t* digest) {
  CTX_CHECK(ctx);
  if (!digest) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n == 0) { CUDA_TRY(ctx, cudaMemsetAsync(digest, 0, sizeof(uint64_t), ctx->compute)); return PBH_OK; }
  if (!wit || !rnd || !proof || !status) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || proof_pitch < n || (chal_out && chal_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  ProveFsArgs F{{wit, wit_pitch, rnd, rand_pitch, nullptr, 0, proof, proof_pitch, status, n}, chal_out, chal_pitch};
  return launch_prove_fs(ctx, ctx->compute, F, first_index, digest);
}
int pbh_verify_fs_bitmap_batch_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result, uint8_t* bitmap) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !result || !bitmap) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  VerifyFsArgs F{{proof, proof_pitch, nullptr, 0, nullptr, result, nullptr, 0, n, bitmap}, nullptr, 0};
  return launch_verify_fs(ctx, ctx->compute, F);
}
int pbh_prove_fs_batch(pbh_ctx* ctx, size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch,
                       uint8_t* proof, size_t proof_pitch, uint8_t* status, uint8_t* chal_out, size_t chal_pitch) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !proof || !status) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || proof_pitch < n || (chal_out && chal_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    uint8_t *d_wit = at_row(base, C, PR::wit), *d_rnd = at_row(base, C, PR::rnd), *d_proof = at_row(base, C, PR::proof),
            *d_status = at_row(base, C, PR::status), *d_chal = at_row(base, C, FsRows::chal_out);
    PBH_TRY(stage_h2d(ctx, base, st, d_wit, C, wit + lo, wit_pitch, m, PR::wit.count));
    PBH_TRY(stage_h2d(ctx, base, st, d_rnd, C, rnd + lo, rand_pitch, m, PR::rnd.count));
    ProveFsArgs F{{d_wit, C, d_rnd, C, nullptr, 0, d_proof, C, d_status, m}, chal_out ? d_chal : nullptr, C};
    int rc = launch_prove_fs(ctx, st, F);
    if (rc) return rc;
    PBH_TRY(stage_d2h(ctx, base, st, proof + lo, proof_pitch, d_proof, C, m, PR::proof.count));
    PBH_TRY(stage_d2h(ctx, base, st, status + lo, 0, d_status, 0, m, 1));
    if (chal_out) PBH_TRY(stage_d2h(ctx, base, st, chal_out + lo, chal_pitch, d_chal, C, m, FsRows::chal_out.count));
    return PBH_OK;
  });
}
int pbh_verify_fs_batch(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, uint8_t* result, uint8_t* chal_out,
                        size_t chal_pitch, uint8_t* gt, size_t gt_pitch) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (proof_pitch < n || (chal_out && chal_pitch < n) || (gt && gt_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    uint8_t *d_proof = at_row(base, C, VR::proof), *d_res = at_row(base, C, VR::res), *d_chal = at_row(base, C, FsRows::chal_out),
            *d_gt = at_row(base, C, VR::gt);
    PBH_TRY(stage_h2d(ctx, base, st, d_proof, C, proof + lo, proof_pitch, m, VR::proof.count));
    VerifyFsArgs F{{d_proof, C, nullptr, 0, nullptr, d_res, gt ? d_gt : nullptr, C, m, nullptr}, chal_out ? d_chal : nullptr, C};
    int rc = launch_verify_fs(ctx, st, F);
    if (rc) return rc;
    PBH_TRY(stage_d2h(ctx, base, st, result + lo, 0, d_res, 0, m, 1));
    if (chal_out) PBH_TRY(stage_d2h(ctx, base, st, chal_out + lo, chal_pitch, d_chal, C, m, FsRows::chal_out.count));
    if (gt) PBH_TRY(stage_d2h(ctx, base, st, gt + lo, gt_pitch, d_gt, C, m, VR::gt.count));
    return PBH_OK;
  });
}

// ---- record wire format ------------------------------------------------------------------------------------------
static_assert(sizeof(pbh_witness_record) == 32 && sizeof(pbh_proof_record) == 32, "records are 32 bytes");

int pbh_witness_records_to_planes_dev(pbh_ctx* ctx, size_t n, const pbh_witness_record* rec, uint8_t* wit, size_t wit_pitch, uint8_t* rnd,
                                      size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!rec || ((uintptr_t)rec % 16) != 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "records must be 16-byte aligned");
  if ((wit && wit_pitch < n) || (rnd && rand_pitch < n) || (chal && chal_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  witness_records_to_planes_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(n, rec, wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, u);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}
int pbh_proof_records_to_planes_dev(pbh_ctx* ctx, size_t n, const pbh_proof_record* rec, uint8_t* proof, size_t proof_pitch, uint8_t* status) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!rec || ((uintptr_t)rec % 16) != 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "records must be 16-byte aligned");
  if (proof && proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  proof_records_to_planes_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(n, rec, proof, proof_pitch, status);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}
int pbh_proof_planes_to_records_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status,
                                    pbh_proof_record* rec) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!rec || !proof || ((uintptr_t)rec % 16) != 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer or records not 16-byte aligned");
  if (proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  proof_planes_to_records_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(n, proof, proof_pitch, status, rec);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}

// host records: per chunk, H2D records -> transpose -> plane kernels -> transpose -> D2H records, over the staging slots
int pbh_prove_records(pbh_ctx* ctx, size_t n, const pbh_witness_record* in, pbh_proof_record* out) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!in || !out) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    uint8_t *d_wit = at_row(base, C, PR::wit), *d_rnd = at_row(base, C, PR::rnd), *d_chal = at_row(base, C, PR::chal),
            *d_proof = at_row(base, C, PR::proof), *d_status = at_row(base, C, PR::status);
    pbh_witness_record* d_in = at_row<pbh_witness_record>(base, C, RecordRows::witness);
    pbh_proof_record* d_out = at_row<pbh_proof_record>(base, C, RecordRows::proof);
    PBH_TRY(stage_h2d(ctx, base, st, d_in, 0, in + lo, 0, m * sizeof(pbh_witness_record), 1));
    witness_records_to_planes_kernel<<<grid_for(ctx, m, 8), kBlock, 0, st>>>(m, d_in, d_wit, C, d_rnd, C, d_chal, C, nullptr);
    ctx->launches++;
    ProveArgs A{d_wit, C, d_rnd, C, d_chal, C, d_proof, C, d_status, m};
    int rc = launch_prove(ctx, st, A);
    if (rc) return rc;
    proof_planes_to_records_kernel<<<grid_for(ctx, m, 8), kBlock, 0, st>>>(m, d_proof, C, d_status, d_out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    PBH_TRY(stage_d2h(ctx, base, st, out + lo, 0, d_out, 0, m * sizeof(pbh_proof_record), 1));
    return PBH_OK;
  });
}

int pbh_verify_records(pbh_ctx* ctx, size_t n, const pbh_proof_record* proofs, const pbh_witness_record* params, uint8_t* result) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proofs || !params || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    uint8_t *d_proof = at_row(base, C, VR::proof), *d_chal = at_row(base, C, VR::chal), *d_u = at_row(base, C, VR::u);
    pbh_witness_record* d_par = at_row<pbh_witness_record>(base, C, RecordRows::witness);
    pbh_proof_record* d_prf = at_row<pbh_proof_record>(base, C, RecordRows::proof);
    PBH_TRY(stage_h2d(ctx, base, st, d_prf, 0, proofs + lo, 0, m * sizeof(pbh_proof_record), 1));
    PBH_TRY(stage_h2d(ctx, base, st, d_par, 0, params + lo, 0, m * sizeof(pbh_witness_record), 1));
    proof_records_to_planes_kernel<<<grid_for(ctx, m, 8), kBlock, 0, st>>>(m, d_prf, d_proof, C, nullptr);
    witness_records_to_planes_kernel<<<grid_for(ctx, m, 8), kBlock, 0, st>>>(m, d_par, nullptr, 0, nullptr, 0, d_chal, C, d_u);
    ctx->launches += 2;
    return verify_body(ctx, st, base, C, VerifyArgs{d_proof, C, d_chal, C, d_u, result + lo, nullptr, 0, m, nullptr}, false, true);
  });
}

// ---- packed wire format (include/pbh_b200.h "packed wire format", csrc/pbh_packed.cuh) ------------------------------------
static_assert(sizeof(pbh_packed_witness) == 16 && sizeof(pbh_packed_proof) == 12, "packed records are 16 and 12 bytes");
static int launch_unpack_witness(pbh_ctx* ctx, cudaStream_t st, size_t n, const pbh_packed_witness* in, uint8_t* wit, size_t wit_pitch,
                                 uint8_t* rnd, size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u) {
  auto al4 = [](const void* p, size_t pitch) { return !p || (((uintptr_t)p | pitch) % 4) == 0; };
  const bool vec = al4(wit, wit_pitch) && al4(rnd, rand_pitch) && al4(chal, chal_pitch) && al4(u, 0);
  unpack_witness_kernel<<<grid_for(ctx, (n + 3) / 4, 8), kBlock, 0, st>>>(n, in, wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, u, vec);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}
static int launch_pack_proof(pbh_ctx* ctx, cudaStream_t st, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status,
                             pbh_packed_proof* out) {
  const bool vec = (((uintptr_t)proof | proof_pitch) % 4) == 0 && ((uintptr_t)status % 4) == 0 && ((uintptr_t)out % 16) == 0;
  pack_proof_kernel<<<grid_for(ctx, (n + 3) / 4, 8), kBlock, 0, st>>>(n, proof, proof_pitch, status, out, vec);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}
static int launch_unpack_proof(pbh_ctx* ctx, cudaStream_t st, size_t n, const pbh_packed_proof* in, const uint32_t* chal_u, uint8_t* proof,
                               size_t proof_pitch, uint8_t* status, uint8_t* chal, size_t chal_pitch, uint8_t* u) {
  auto al4 = [](const void* p, size_t pitch) { return !p || (((uintptr_t)p | pitch) % 4) == 0; };
  const bool vec = al4(proof, proof_pitch) && al4(status, 0) && al4(chal, chal_pitch) && al4(u, 0) && ((uintptr_t)in % 16) == 0;
  unpack_proof_kernel<<<grid_for(ctx, (n + 3) / 4, 8), kBlock, 0, st>>>(n, in, chal_u, proof, proof_pitch, status, chal, chal_pitch, u, vec);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}

int pbh_unpack_witness_dev(pbh_ctx* ctx, size_t n, const pbh_packed_witness* in, uint8_t* wit, size_t wit_pitch, uint8_t* rnd,
                           size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!in || ((uintptr_t)in % 16) != 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "packed witnesses must be 16-byte aligned");
  if ((wit && wit_pitch < n) || (rnd && rand_pitch < n) || (chal && chal_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return launch_unpack_witness(ctx, ctx->compute, n, in, wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, u);
}
int pbh_pack_proof_dev(pbh_ctx* ctx, size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status, pbh_packed_proof* out) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proof || !out || ((uintptr_t)out % 4) != 0) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer or packed proofs not 4-byte aligned");
  if (proof_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return launch_pack_proof(ctx, ctx->compute, n, proof, proof_pitch, status, out);
}
int pbh_unpack_proof_dev(pbh_ctx* ctx, size_t n, const pbh_packed_proof* in, const uint32_t* chal_u, uint8_t* proof, size_t proof_pitch,
                         uint8_t* status, uint8_t* chal, size_t chal_pitch, uint8_t* u) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if ((!in && !chal_u) || ((uintptr_t)in % 4) != 0 || ((uintptr_t)chal_u % 4) != 0)
    return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointers or packed words not 4-byte aligned");
  if ((in && !proof) || (proof && proof_pitch < n) || (chal && chal_pitch < n)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "proof planes missing or pitch < n");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return launch_unpack_proof(ctx, ctx->compute, n, in, chal_u, proof, proof_pitch, status, chal, chal_pitch, u);
}

// One chunk (or one whole lane batch) of the packed prover / verifier on stream st, staged in `base` (PackedRows).
static int packed_prove_body(pbh_ctx* ctx, cudaStream_t st, uint8_t* base, size_t C, size_t m, const pbh_packed_witness* in,
                             pbh_packed_proof* out, uint8_t* result_host) {
  uint8_t *d_wit = at_row(base, C, PR::wit), *d_rnd = at_row(base, C, PR::rnd), *d_chal = at_row(base, C, PR::chal),
          *d_proof = at_row(base, C, PR::proof), *d_status = at_row(base, C, PR::status), *d_u = at_row(base, C, PR::u),
          *d_res = at_row(base, C, PR::res);
  pbh_packed_witness* d_in = at_row<pbh_packed_witness>(base, C, PackedRows::in);
  pbh_packed_proof* d_out = at_row<pbh_packed_proof>(base, C, PackedRows::out);
  PBH_TRY(stage_h2d(ctx, base, st, d_in, 0, in, 0, m * sizeof(pbh_packed_witness), 1));
  int rc = launch_unpack_witness(ctx, st, m, d_in, d_wit, C, d_rnd, C, d_chal, C, result_host ? d_u : nullptr);
  if (rc) return rc;
  ProveArgs A{d_wit, C, d_rnd, C, d_chal, C, d_proof, C, d_status, m};
  rc = launch_prove(ctx, st, A);
  if (rc) return rc;
  if (result_host) {
    VerifyArgs V{d_proof, C, d_chal, C, d_u, d_res, nullptr, 0, m, nullptr};
    rc = launch_verify(ctx, st, V);
    if (rc) return rc;
  }
  rc = launch_pack_proof(ctx, st, m, d_proof, C, d_status, d_out);
  if (rc) return rc;
  PBH_TRY(stage_d2h(ctx, base, st, out, 0, d_out, 0, m * sizeof(pbh_packed_proof), 1));
  if (result_host) PBH_TRY(stage_d2h(ctx, base, st, result_host, 0, d_res, 0, m, 1));
  return PBH_OK;
}
// `resident`: the proof planes these packed proofs decode to are already at rows VR::proof of `base` - the prove call that produced
// `proofs` on this lane left them there (packed_prove_body), and pack -> unpack is the identity on a prover's output - so neither
// the upload of the proofs nor their decoding is repeated; only the challenge words travel.
static int packed_verify_body(pbh_ctx* ctx, cudaStream_t st, uint8_t* base, size_t C, size_t m, const pbh_packed_proof* proofs,
                              const uint32_t* chal_u, uint8_t* result, bool resident = false) {
  uint8_t *d_proof = at_row(base, C, VR::proof), *d_chal = at_row(base, C, VR::chal), *d_u = at_row(base, C, VR::u);
  pbh_packed_proof* d_prf = at_row<pbh_packed_proof>(base, C, PackedRows::proofs);
  uint32_t* d_cu = at_row<uint32_t>(base, C, PackedRows::chal_u);
  if (!resident) PBH_TRY(stage_h2d(ctx, base, st, d_prf, 0, proofs, 0, m * sizeof(pbh_packed_proof), 1));
  PBH_TRY(stage_h2d(ctx, base, st, d_cu, 0, chal_u, 0, m * sizeof(uint32_t), 1));
  PBH_TRY(launch_unpack_proof(ctx, st, m, resident ? nullptr : d_prf, d_cu, d_proof, C, nullptr, d_chal, C, d_u));
  return verify_body(ctx, st, base, C, VerifyArgs{d_proof, C, d_chal, C, d_u, result, nullptr, 0, m, nullptr}, false, true);
}

int pbh_prove_packed(pbh_ctx* ctx, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!in || !out) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    return packed_prove_body(ctx, st, base, C, m, in + lo, out + lo, nullptr);
  });
}
int pbh_prove_verify_packed(pbh_ctx* ctx, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out, uint8_t* result) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!in || !out || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    return packed_prove_body(ctx, st, base, C, m, in + lo, out + lo, result + lo);
  });
}
int pbh_verify_packed(pbh_ctx* ctx, size_t n, const pbh_packed_proof* proofs, const uint32_t* chal_u, uint8_t* result) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proofs || !chal_u || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    return packed_verify_body(ctx, st, base, C, m, proofs + lo, chal_u + lo, result + lo);
  });
}
int pbh_prove_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out) {
  CTX_CHECK(ctx);
  return lane_call(ctx, lane, n, !in || !out ? "null pointer" : nullptr, [&] { return staged_plan(n, PackedRows::kProveRows, {in, out}); },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void*) -> int {
        PBH_TRY(packed_prove_body(ctx, st, base, C, n, in, out, nullptr));
        if (ctx->proof_resident) { ctx->resident_host[lane] = out; ctx->resident_n[lane] = n; }
        return PBH_OK;
      },
      [&] { return pbh_prove_packed(ctx, n, in, out); });
}
int pbh_prove_verify_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_witness* in, pbh_packed_proof* out, uint8_t* result) {
  CTX_CHECK(ctx);
  return lane_call(ctx, lane, n, !in || !out || !result ? "null pointer" : nullptr,
      [&] { return staged_plan(n, PackedRows::kProveRows, {in, out, result}); },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void*) { return packed_prove_body(ctx, st, base, C, n, in, out, result); },
      [&] { return pbh_prove_verify_packed(ctx, n, in, out, result); });
}
int pbh_verify_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_proof* proofs, const uint32_t* chal_u, uint8_t* result) {
  CTX_CHECK(ctx);
  return lane_call(ctx, lane, n, !proofs || !chal_u || !result ? "null pointer" : nullptr,
      [&] { return staged_plan(n, PackedRows::kVerifyRows, {proofs, chal_u, result}); },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void* resident) {
        // the very buffer the previous call on this lane is still filling, with no synchronisation in between (the caller may not
        // touch it before pbh_lane_sync): its contents ARE the proofs resident in the lane buffer
        return packed_verify_body(ctx, st, base, C, n, proofs, chal_u, result, ctx->proof_resident && resident == proofs);
      },
      [&] { return pbh_verify_packed(ctx, n, proofs, chal_u, result); });
}

// host-side format conversion: the codec of pbh_packed.cuh on the CPU (no context, no device)
int pbh_pack_witness_host(size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch, const uint8_t* chal,
                          size_t chal_pitch, const uint8_t* u, pbh_packed_witness* out) {
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !out || wit_pitch < n || rand_pitch < n || (chal && chal_pitch < n)) return PBH_ERR_BAD_ARGUMENT;
  bool ok = true;
  for (size_t i = 0; i < n; i++) {
    uint8_t v[27];
    for (int k = 0; k < 12; k++) v[k] = wit[k * wit_pitch + i];
    for (int k = 0; k < 9; k++) v[12 + k] = rnd[k * rand_pitch + i];
    for (int k = 0; k < 5; k++) v[21 + k] = chal ? chal[k * chal_pitch + i] : 0;
    v[26] = u ? u[i] : 0;
    ok = pack_witness_item(v, out[i].w) && ok;
  }
  return ok ? PBH_OK : PBH_ERR_BAD_ARGUMENT;
}
int pbh_unpack_witness_host(size_t n, const pbh_packed_witness* in, uint8_t* wit, size_t wit_pitch, uint8_t* rnd, size_t rand_pitch,
                            uint8_t* chal, size_t chal_pitch, uint8_t* u) {
  if (n == 0) return PBH_OK;
  if (!in || (wit && wit_pitch < n) || (rnd && rand_pitch < n) || (chal && chal_pitch < n)) return PBH_ERR_BAD_ARGUMENT;
  for (size_t i = 0; i < n; i++) {
    uint8_t v[27];
    unpack_witness_item(in[i].w, v);
    if (wit) for (int k = 0; k < 12; k++) wit[k * wit_pitch + i] = v[k];
    if (rnd) for (int k = 0; k < 9; k++) rnd[k * rand_pitch + i] = v[12 + k];
    if (chal) for (int k = 0; k < 5; k++) chal[k * chal_pitch + i] = v[21 + k];
    if (u) u[i] = v[26];
  }
  return PBH_OK;
}
int pbh_pack_chal_u_host(size_t n, const uint8_t* chal, size_t chal_pitch, const uint8_t* u, uint32_t* out) {
  if (n == 0) return PBH_OK;
  if (!chal || !u || !out || chal_pitch < n) return PBH_ERR_BAD_ARGUMENT;
  bool ok = true;
  for (size_t i = 0; i < n; i++) {
    uint8_t v[6];
    for (int k = 0; k < 5; k++) v[k] = chal[k * chal_pitch + i];
    v[5] = u[i];
    ok = pack_chal_u(v, &out[i]) && ok;
  }
  return ok ? PBH_OK : PBH_ERR_BAD_ARGUMENT;
}
int pbh_pack_proofs_host(size_t n, const uint8_t* proof, size_t proof_pitch, const uint8_t* status, pbh_packed_proof* out) {
  if (n == 0) return PBH_OK;
  if (!proof || !out || proof_pitch < n) return PBH_ERR_BAD_ARGUMENT;
  for (size_t i = 0; i < n; i++) {
    uint8_t p[27];
    for (int k = 0; k < 27; k++) p[k] = proof[k * proof_pitch + i];
    uint32_t w[3];
    pack_proof_item(kPackedTablesHost, p, status ? status[i] : (uint8_t)0, w);
    out[i].points_lo = w[0]; out[i].points_hi = w[1]; out[i].evals_status = w[2];
  }
  return PBH_OK;
}
int pbh_unpack_proofs_host(size_t n, const pbh_packed_proof* in, uint8_t* proof, size_t proof_pitch, uint8_t* status) {
  if (n == 0) return PBH_OK;
  if (!in || (proof && proof_pitch < n)) return PBH_ERR_BAD_ARGUMENT;
  for (size_t i = 0; i < n; i++) {
    const uint32_t w[3] = {in[i].points_lo, in[i].points_hi, in[i].evals_status};
    uint8_t p[27], st;
    unpack_proof_item(kPackedTablesHost, w, p, &st);
    if (proof) for (int k = 0; k < 27; k++) proof[k * proof_pitch + i] = p[k];
    if (status) status[i] = st;
  }
  return PBH_OK;
}

// ---- Fiat-Shamir over packed records (include/pbh_b200.h) ---------------------------------------------------------------------
static_assert(sizeof(pbh_packed_fs_witness) == 12, "packed Fiat-Shamir witnesses are 12 bytes");
static int launch_prove_fs_packed(pbh_ctx* ctx, cudaStream_t st, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out,
                                  uint32_t* chal_u_out) {
  if (n == 0) return PBH_OK;
  const int grid = grid_for(ctx, n, 2);
  const FsSeed seed = fs_seed_of(ctx);
  const uint32_t* i32 = reinterpret_cast<const uint32_t*>(in);
  uint32_t* o32 = reinterpret_cast<uint32_t*>(out);
  with_fs_prover(ctx, [&](auto P) {
    using I = decltype(P);
    prove_fs_packed_kernel<I::algo, I::fp32, I::pbh_circuit><<<grid, 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, seed, ctx->d_tables, n, i32, o32, chal_u_out);
  });
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}
static int launch_verify_fs_packed(pbh_ctx* ctx, cudaStream_t st, size_t n, const pbh_packed_proof* proofs, uint8_t* result) {
  if (n == 0) return PBH_OK;
  const int grid = grid_for(ctx, n, 2);
  const FsSeed seed = fs_seed_of(ctx);
  const uint32_t* p32 = reinterpret_cast<const uint32_t*>(proofs);
  with_fs_verifier(ctx, [&](auto algo, bool fp32) {
    verify_fs_packed_kernel<decltype(algo)::value><<<grid, 256, 0, st>>>(ctx->hs.K, ctx->hs.KF, fp32, seed, ctx->d_tables, n, p32, result);
  });
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return PBH_OK;
}
static bool aligned4(const void* p) { return ((uintptr_t)p % 4) == 0; }

int pbh_prove_fs_packed_dev(pbh_ctx* ctx, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!in || !out) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (!aligned4(in) || !aligned4(out) || !aligned4(chal_u_out)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "packed records must be 4-byte aligned");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return launch_prove_fs_packed(ctx, ctx->compute, n, in, out, chal_u_out);
}
int pbh_verify_fs_packed_dev(pbh_ctx* ctx, size_t n, const pbh_packed_proof* proofs, uint8_t* result) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proofs || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (!aligned4(proofs)) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "packed proofs must be 4-byte aligned");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return launch_verify_fs_packed(ctx, ctx->compute, n, proofs, result);
}

// One chunk (or one whole lane batch) on stream st, staged in `base` (FsPackedRows).
static int fs_packed_prove_body(pbh_ctx* ctx, cudaStream_t st, uint8_t* base, size_t C, size_t m, const pbh_packed_fs_witness* in,
                                pbh_packed_proof* out, uint32_t* chal_u_out) {
  pbh_packed_fs_witness* d_in = at_row<pbh_packed_fs_witness>(base, C, FsPackedRows::in);
  pbh_packed_proof* d_out = at_row<pbh_packed_proof>(base, C, FsPackedRows::out);
  uint32_t* d_cu = at_row<uint32_t>(base, C, FsPackedRows::chal_u);
  PBH_TRY(stage_h2d(ctx, base, st, d_in, 0, in, 0, m * sizeof(pbh_packed_fs_witness), 1));
  PBH_TRY(launch_prove_fs_packed(ctx, st, m, d_in, d_out, chal_u_out ? d_cu : nullptr));
  PBH_TRY(stage_d2h(ctx, base, st, out, 0, d_out, 0, m * sizeof(pbh_packed_proof), 1));
  if (chal_u_out) PBH_TRY(stage_d2h(ctx, base, st, chal_u_out, 0, d_cu, 0, m * sizeof(uint32_t), 1));
  return PBH_OK;
}
static int fs_packed_verify_body(pbh_ctx* ctx, cudaStream_t st, uint8_t* base, size_t C, size_t m, const pbh_packed_proof* proofs,
                                 uint8_t* result) {
  pbh_packed_proof* d_prf = at_row<pbh_packed_proof>(base, C, FsPackedRows::proofs);
  uint8_t* d_res = at_row(base, C, FsPackedRows::res);
  PBH_TRY(stage_h2d(ctx, base, st, d_prf, 0, proofs, 0, m * sizeof(pbh_packed_proof), 1));
  PBH_TRY(launch_verify_fs_packed(ctx, st, m, d_prf, d_res));
  PBH_TRY(stage_d2h(ctx, base, st, result, 0, d_res, 0, m, 1));
  return PBH_OK;
}

int pbh_prove_fs_packed(pbh_ctx* ctx, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!in || !out) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    return fs_packed_prove_body(ctx, st, base, C, m, in + lo, out + lo, chal_u_out ? chal_u_out + lo : nullptr);
  });
}
int pbh_verify_fs_packed(pbh_ctx* ctx, size_t n, const pbh_packed_proof* proofs, uint8_t* result) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!proofs || !result) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(ctx, n, [&](size_t lo, size_t m, size_t C, uint8_t* base, cudaStream_t st) -> int {
    return fs_packed_verify_body(ctx, st, base, C, m, proofs + lo, result + lo);
  });
}
int pbh_prove_fs_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_fs_witness* in, pbh_packed_proof* out, uint32_t* chal_u_out) {
  CTX_CHECK(ctx);
  return lane_call(ctx, lane, n, !in || !out ? "null pointer" : nullptr, [&] { return staged_plan(n, FsPackedRows::kProveRows, {in, out, chal_u_out}); },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void*) { return fs_packed_prove_body(ctx, st, base, C, n, in, out, chal_u_out); },
      [&] { return pbh_prove_fs_packed(ctx, n, in, out, chal_u_out); });
}
// No resident-proof shortcut here (PBH_OPT_PROOF_RESIDENT): the verifier uploads the buffer it is handed, whatever ran before.
int pbh_verify_fs_packed_async(pbh_ctx* ctx, int lane, size_t n, const pbh_packed_proof* proofs, uint8_t* result) {
  CTX_CHECK(ctx);
  return lane_call(ctx, lane, n, !proofs || !result ? "null pointer" : nullptr, [&] { return staged_plan(n, FsPackedRows::kVerifyRows, {proofs, result}); },
      [&](cudaStream_t st, uint8_t* base, size_t C, const void*) { return fs_packed_verify_body(ctx, st, base, C, n, proofs, result); },
      [&] { return pbh_verify_fs_packed(ctx, n, proofs, result); });
}

int pbh_pack_fs_witness_host(size_t n, const uint8_t* wit, size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch, pbh_packed_fs_witness* out) {
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !out || wit_pitch < n || rand_pitch < n) return PBH_ERR_BAD_ARGUMENT;
  bool ok = true;
  for (size_t i = 0; i < n; i++) {
    uint8_t v[27] = {0};   // chal and u stay zero: word 3 of the full witness is not part of this record
    for (int k = 0; k < 12; k++) v[k] = wit[k * wit_pitch + i];
    for (int k = 0; k < 9; k++) v[12 + k] = rnd[k * rand_pitch + i];
    uint32_t w[4];
    ok = pack_witness_item(v, w) && ok;
    for (int j = 0; j < 3; j++) out[i].w[j] = w[j];
  }
  return ok ? PBH_OK : PBH_ERR_BAD_ARGUMENT;
}
int pbh_unpack_fs_witness_host(size_t n, const pbh_packed_fs_witness* in, uint8_t* wit, size_t wit_pitch, uint8_t* rnd, size_t rand_pitch) {
  if (n == 0) return PBH_OK;
  if (!in || (wit && wit_pitch < n) || (rnd && rand_pitch < n)) return PBH_ERR_BAD_ARGUMENT;
  for (size_t i = 0; i < n; i++) {
    uint8_t v[21];
    for (int j = 0; j < 3; j++) digits17<7>(in[i].w[j], v + 7 * j);
    if (wit) for (int k = 0; k < 12; k++) wit[k * wit_pitch + i] = v[k];
    if (rnd) for (int k = 0; k < 9; k++) rnd[k * rand_pitch + i] = v[12 + k];
  }
  return PBH_OK;
}

// ---- sweep entry points ---------------------------------------------------------------------------------
// Host-pointer mode stages whole planes through a temporary device allocation (these are per-kernel test and
// benchmark entry points; the hot host-pointer path is pbh_prove_batch / pbh_verify_batch above).
namespace {
struct Staged {
  pbh_ctx* ctx;
  std::vector<void*> allocs;
  explicit Staged(pbh_ctx* c) : ctx(c) {}
  ~Staged() { for (void* p : allocs) cudaFree(p); }
  // returns a device pointer to `planes` planes of pitch n holding a copy of the host planes (or uninitialised)
  template <class T>
  T* in(const T* host, size_t pitch, size_t n, size_t planes, cudaError_t& e) {
    T* d = nullptr;
    e = cudaMalloc((void**)&d, std::max<size_t>(1, planes * n * sizeof(T)));
    if (e != cudaSuccess) return nullptr;
    allocs.push_back(d);
    if (host) e = cudaMemcpy2DAsync(d, n * sizeof(T), host, pitch * sizeof(T), n * sizeof(T), planes, cudaMemcpyHostToDevice, ctx->compute);
    return d;
  }
  template <class T>
  cudaError_t out(T* host, size_t pitch, const T* d, size_t n, size_t planes) {
    return cudaMemcpy2DAsync(host, pitch * sizeof(T), d, n * sizeof(T), n * sizeof(T), planes, cudaMemcpyDeviceToHost, ctx->compute);
  }
};
}  // namespace

#define SWEEP_PROLOGUE(ctx, n)                         \
  CTX_CHECK(ctx);                                      \
  if ((n) == 0) return PBH_OK;                         \
  CUDA_TRY(ctx, cudaSetDevice((ctx)->device));         \
  cudaError_t ce = cudaSuccess;                        \
  (void)ce;                                            \
  Staged stg(ctx)

#define SWEEP_FINISH(ctx)                              \
  (ctx)->launches++;                                   \
  CUDA_TRY(ctx, cudaGetLastError())

static int ntt4_impl(pbh_ctx* ctx, bool inverse, uint32_t k, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch,
                     int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!in || !out || in_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (k < 1 || k > 3) return fail(ctx, PBH_ERR_UNSUPPORTED, "coset shift must be 1 (H), 2 (K1) or 3 (K2): src/pbh/mod.rs:27-28");
  const uint8_t* d_in = in; uint8_t* d_out = out; size_t ip = in_pitch, op = out_pitch;
  if (!on_device) {
    d_in = stg.in(in, in_pitch, n, 4, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint8_t>(nullptr, 0, n, 4, ce); CUDA_TRY(ctx, ce);
    ip = op = n;
  }
  auto aligned = [&](size_t a) { return ((uintptr_t)d_in % a == 0) && ((uintptr_t)d_out % a == 0) && (ip % a == 0) && (op % a == 0); };
  const int vec = aligned(16) ? 16 : (aligned(4) ? 4 : 0);
  int grid = grid_for(ctx, vec ? (n + vec - 1) / vec : n, 8);
#define PBH_NTT4(INV, KK) ntt4_kernel<INV, KK><<<grid, kBlock, 0, ctx->compute>>>(n, d_in, ip, d_out, op, vec)
  if (inverse) { if (k == 1) PBH_NTT4(true, 1); else if (k == 2) PBH_NTT4(true, 2); else PBH_NTT4(true, 3); }
  else { if (k == 1) PBH_NTT4(false, 1); else if (k == 2) PBH_NTT4(false, 2); else PBH_NTT4(false, 3); }
#undef PBH_NTT4
  SWEEP_FINISH(ctx);
  if (!on_device) { CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, 4)); CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute)); }
  return PBH_OK;
}
int pbh_ntt4_batch(pbh_ctx* ctx, size_t n, const uint8_t* coeffs, size_t in_pitch, uint8_t* evals, size_t out_pitch, int on_device) {
  return ntt4_impl(ctx, false, 1, n, coeffs, in_pitch, evals, out_pitch, on_device);
}
int pbh_intt4_batch(pbh_ctx* ctx, size_t n, const uint8_t* evals, size_t in_pitch, uint8_t* coeffs, size_t out_pitch, int on_device) {
  return ntt4_impl(ctx, true, 1, n, evals, in_pitch, coeffs, out_pitch, on_device);
}
int pbh_coset_ntt4_batch(pbh_ctx* ctx, size_t n, uint32_t k, const uint8_t* coeffs, size_t in_pitch, uint8_t* evals, size_t out_pitch,
                         int on_device) {
  return ntt4_impl(ctx, false, k, n, coeffs, in_pitch, evals, out_pitch, on_device);
}
int pbh_coset_intt4_batch(pbh_ctx* ctx, size_t n, uint32_t k, const uint8_t* evals, size_t in_pitch, uint8_t* coeffs, size_t out_pitch,
                          int on_device) {
  return ntt4_impl(ctx, true, k, n, evals, in_pitch, coeffs, out_pitch, on_device);
}

int pbh_ntt_generic_batch(pbh_ctx* ctx, size_t n, uint32_t modulus, uint32_t omega, uint32_t size, int inverse, const uint16_t* in,
                          size_t in_pitch, uint16_t* out, size_t out_pitch, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!in || !out || in_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (modulus < 2 || modulus >= 65536 || size < 2 || size > 64 || (size & (size - 1))) return fail(ctx, PBH_ERR_UNSUPPORTED, "modulus < 2^16, size a power of two in [2, 64]");
  uint32_t log2size = 0;
  while ((1u << log2size) < size) log2size++;
  // twiddles omega^i (CooleyTurkey::new, src/fft.rs:52-64) and size^-1 by Fermat (modulus prime, as in the reference's tests)
  uint16_t tw[64];
  uint32_t m = 1;
  for (uint32_t i = 0; i < size; i++) { tw[i] = (uint16_t)m; m = (uint32_t)(((uint64_t)m * (omega % modulus)) % modulus); }
  uint64_t len_inv = 1, b = size % modulus, e = modulus - 2;
  while (e) { if (e & 1) len_inv = len_inv * b % modulus; b = b * b % modulus; e >>= 1; }
  // only fft_inv asks for the length inverse (src/fft.rs:72-78): the forward transform exists for every modulus
  if (inverse && (len_inv * (size % modulus)) % modulus != 1)
    return fail(ctx, PBH_ERR_SETUP_PANIC, "size has no inverse modulo the modulus (F::from(len).inv().unwrap() panics)");
  uint16_t* d_tw = stg.in(tw, 64, 64, 1, ce); CUDA_TRY(ctx, ce);
  const uint16_t* d_in = in; uint16_t* d_out = out; size_t ip = in_pitch, op = out_pitch;
  if (!on_device) {
    d_in = stg.in(in, in_pitch, n, size, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint16_t>(nullptr, 0, n, size, ce); CUDA_TRY(ctx, ce);
    ip = op = n;
  }
  ntt_generic_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(n, modulus, size, log2size, (uint32_t)len_inv, inverse, d_tw, d_in, ip, d_out, op);
  SWEEP_FINISH(ctx);
  if (!on_device) CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, size));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute));   // d_tw is freed on return
  return PBH_OK;
}

int pbh_mul_ntt_batch(pbh_ctx* ctx, size_t n, uint32_t modulus, uint32_t omega, uint32_t la, uint32_t lb, const uint16_t* a,
                      size_t a_pitch, const uint16_t* b, size_t b_pitch, uint16_t* out, size_t out_pitch, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!a || !b || !out || a_pitch < n || b_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  const uint32_t size = la + lb;
  if (la < 1 || lb < 1 || modulus < 2 || modulus >= 65536 || size < 2 || size > 64 || (size & (size - 1)))
    return fail(ctx, PBH_ERR_UNSUPPORTED, "modulus < 2^16, la + lb a power of two in [2, 64]");
  uint32_t log2size = 0;
  while ((1u << log2size) < size) log2size++;
  uint16_t tw[64];
  uint32_t m = 1;
  for (uint32_t i = 0; i < size; i++) { tw[i] = (uint16_t)m; m = (uint32_t)(((uint64_t)m * (omega % modulus)) % modulus); }
  uint64_t len_inv = 1, bb = size % modulus, e = modulus - 2;
  while (e) { if (e & 1) len_inv = len_inv * bb % modulus; bb = bb * bb % modulus; e >>= 1; }
  if ((len_inv * (size % modulus)) % modulus != 1) return fail(ctx, PBH_ERR_SETUP_PANIC, "size has no inverse modulo the modulus (F::from(len).inv().unwrap() panics)");
  uint16_t* d_tw = stg.in(tw, 64, 64, 1, ce); CUDA_TRY(ctx, ce);
  const uint16_t *d_a = a, *d_b = b; uint16_t* d_out = out; size_t ap = a_pitch, bp = b_pitch, op = out_pitch;
  if (!on_device) {
    d_a = stg.in(a, a_pitch, n, la, ce); CUDA_TRY(ctx, ce);
    d_b = stg.in(b, b_pitch, n, lb, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint16_t>(nullptr, 0, n, size, ce); CUDA_TRY(ctx, ce);
    ap = bp = op = n;
  }
  mul_ntt_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(n, modulus, size, log2size, (uint32_t)len_inv, la, lb, d_tw, d_a, ap, d_b, bp, d_out, op);
  SWEEP_FINISH(ctx);
  if (!on_device) CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, size));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute));   // d_tw is freed on return
  return PBH_OK;
}

// len coefficient planes + one operand plane in; OP 0 scale (len planes out), 1 eval (1 plane), 2 divide by x - c (len planes)
template <int OP>
static int poly_unary_impl(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch,
                           int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!in || !out || in_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (len < 1 || len > 64) return fail(ctx, PBH_ERR_UNSUPPORTED, "1 <= len <= 64");
  const size_t pout = OP == 1 ? 1 : len;
  const uint8_t* d_in = in; uint8_t* d_out = out; size_t ip = in_pitch, op = out_pitch;
  if (!on_device) {
    d_in = stg.in(in, in_pitch, n, len + 1, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint8_t>(nullptr, 0, n, pout, ce); CUDA_TRY(ctx, ce);
    ip = op = n;
  }
  // eval writes one plane, so its output pitch (n, see pbh_poly_eval_batch) must not decide the access width
  auto aligned = [&](size_t a) { return ((uintptr_t)d_in % a == 0) && ((uintptr_t)d_out % a == 0) && (ip % a == 0) && (pout == 1 || op % a == 0); };
  const int vec = aligned(16) ? 16 : (aligned(4) ? 4 : 0);
  poly_unary_kernel<OP><<<grid_for(ctx, vec ? (n + vec - 1) / vec : n, 8), kBlock, 0, ctx->compute>>>(n, len, d_in, ip, d_out, op, vec);
  SWEEP_FINISH(ctx);
  if (!on_device) { CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, pout)); CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute)); }
  return PBH_OK;
}
int pbh_poly_scale_batch(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return poly_unary_impl<0>(ctx, n, len, in, in_pitch, out, out_pitch, on_device);
}
int pbh_poly_eval_batch(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, int on_device) {
  return poly_unary_impl<1>(ctx, n, len, in, in_pitch, out, n, on_device);
}
int pbh_poly_div_linear_batch(pbh_ctx* ctx, size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return poly_unary_impl<2>(ctx, n, len, in, in_pitch, out, out_pitch, on_device);
}

int pbh_poly_mul_batch(pbh_ctx* ctx, size_t n, uint32_t la, uint32_t lb, const uint8_t* a, size_t a_pitch, const uint8_t* b,
                       size_t b_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!a || !b || !out || a_pitch < n || b_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (la < 1 || lb < 1 || la > 16 || lb > 16) return fail(ctx, PBH_ERR_UNSUPPORTED, "1 <= la, lb <= 16");
  const uint8_t *d_a = a, *d_b = b; uint8_t* d_out = out; size_t ap = a_pitch, bp = b_pitch, op = out_pitch;
  if (!on_device) {
    d_a = stg.in(a, a_pitch, n, la, ce); CUDA_TRY(ctx, ce);
    d_b = stg.in(b, b_pitch, n, lb, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint8_t>(nullptr, 0, n, la + lb - 1, ce); CUDA_TRY(ctx, ce);
    ap = bp = op = n;
  }
  // operands up to 8 coefficients, 4-byte aligned planes: four items per word in the size-specialised FP32 kernel; the
  // ragged tail (n % 4 items) and everything else go through the general kernel
  const bool vec_ok = la <= 8 && lb <= 8 && ((uintptr_t)d_a % 4 == 0) && ((uintptr_t)d_b % 4 == 0) && ((uintptr_t)d_out % 4 == 0) && (ap % 4 == 0) &&
                      (bp % 4 == 0) && (op % 4 == 0);
  const size_t n4 = vec_ok ? n / 4 : 0;
  if (n4) {
    const int grid = grid_for(ctx, n4, 8);
#define PBH_MUL_CASE(LA, LB) poly_mul_vec_kernel<LA, LB><<<grid, kBlock, 0, ctx->compute>>>(n4, la, lb, d_a, ap, d_b, bp, d_out, op)
#define PBH_MUL_ROW(LA)                                                                     \
    switch ((lb + 1) / 2) { case 1: PBH_MUL_CASE(LA, 2); break; case 2: PBH_MUL_CASE(LA, 4); break; \
                            case 3: PBH_MUL_CASE(LA, 6); break; default: PBH_MUL_CASE(LA, 8); break; }
    switch ((la + 1) / 2) {
      case 1: PBH_MUL_ROW(2); break;
      case 2: PBH_MUL_ROW(4); break;
      case 3: PBH_MUL_ROW(6); break;
      default: PBH_MUL_ROW(8); break;
    }
#undef PBH_MUL_ROW
#undef PBH_MUL_CASE
    ctx->launches++;
  }
  if (n4 * 4 < n) poly_mul_kernel<<<grid_for(ctx, n - n4 * 4, 8), kBlock, 0, ctx->compute>>>(n - n4 * 4, la, lb, d_a + n4 * 4, ap, d_b + n4 * 4, bp, d_out + n4 * 4, op);
  else ctx->launches--;   // SWEEP_FINISH counts one launch
  SWEEP_FINISH(ctx);
  if (!on_device) { CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, la + lb - 1)); CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute)); }
  return PBH_OK;
}

int pbh_poly_add_batch(pbh_ctx* ctx, size_t n, uint32_t len, int subtract, const uint8_t* a, size_t a_pitch, const uint8_t* b,
                       size_t b_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!a || !b || !out || a_pitch < n || b_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (len < 1 || len > 64) return fail(ctx, PBH_ERR_UNSUPPORTED, "1 <= len <= 64");
  const uint8_t *d_a = a, *d_b = b; uint8_t* d_out = out; size_t ap = a_pitch, bp = b_pitch, op = out_pitch;
  if (!on_device) {
    d_a = stg.in(a, a_pitch, n, len, ce); CUDA_TRY(ctx, ce);
    d_b = stg.in(b, b_pitch, n, len, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint8_t>(nullptr, 0, n, len, ce); CUDA_TRY(ctx, ce);
    ap = bp = op = n;
  }
  const bool vec_ok = ((uintptr_t)d_a % 4 == 0) && ((uintptr_t)d_b % 4 == 0) && ((uintptr_t)d_out % 4 == 0) && (ap % 4 == 0) && (bp % 4 == 0) &&
                      (op % 4 == 0);
  poly_add_kernel<<<grid_for(ctx, vec_ok ? (n + 3) / 4 : n, 16), kBlock, 0, ctx->compute>>>(n, len, subtract, d_a, ap, d_b, bp, d_out, op, vec_ok);
  SWEEP_FINISH(ctx);
  if (!on_device) { CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, len)); CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute)); }
  return PBH_OK;
}

int pbh_poly_div_zh_batch(pbh_ctx* ctx, size_t n, const uint8_t* p, size_t p_pitch, uint8_t* q, size_t q_pitch, uint8_t* r,
                          size_t r_pitch, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!p || !q || !r || p_pitch < n || q_pitch < n || r_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  const uint8_t* d_p = p; uint8_t *d_q = q, *d_r = r; size_t pp = p_pitch, qp = q_pitch, rp = r_pitch;
  if (!on_device) {
    d_p = stg.in(p, p_pitch, n, 22, ce); CUDA_TRY(ctx, ce);
    d_q = stg.in<uint8_t>(nullptr, 0, n, 18, ce); CUDA_TRY(ctx, ce);
    d_r = stg.in<uint8_t>(nullptr, 0, n, 4, ce); CUDA_TRY(ctx, ce);
    pp = qp = rp = n;
  }
  const bool vec_ok = ((uintptr_t)d_p % 4 == 0) && ((uintptr_t)d_q % 4 == 0) && ((uintptr_t)d_r % 4 == 0) && (pp % 4 == 0) && (qp % 4 == 0) &&
                      (rp % 4 == 0);
  poly_div_zh_kernel<<<grid_for(ctx, vec_ok ? (n + 3) / 4 : n, 16), kBlock, 0, ctx->compute>>>(n, d_p, pp, d_q, qp, d_r, rp, vec_ok);
  SWEEP_FINISH(ctx);
  if (!on_device) {
    CUDA_TRY(ctx, stg.out(q, q_pitch, d_q, n, 18));
    CUDA_TRY(ctx, stg.out(r, r_pitch, d_r, n, 4));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute));
  }
  return PBH_OK;
}

// common shape: `pin` input planes -> `pout` output planes, kernel(gT, n, in, ip, out, op)
template <class Launch>
static int planes_impl(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, size_t pin, uint8_t* out, size_t out_pitch,
                       size_t pout, int on_device, Launch launch) {
  SWEEP_PROLOGUE(ctx, n);
  if (!in || !out || in_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  const uint8_t* d_in = in; uint8_t* d_out = out; size_t ip = in_pitch, op = out_pitch;
  if (!on_device) {
    d_in = stg.in(in, in_pitch, n, pin, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint8_t>(nullptr, 0, n, pout, ce); CUDA_TRY(ctx, ce);
    ip = op = n;
  }
  launch(grid_for(ctx, n, 8), d_in, ip, d_out, op);
  SWEEP_FINISH(ctx);
  if (!on_device) { CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, pout)); CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute)); }
  return PBH_OK;
}

int pbh_g1_smul_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return planes_impl(ctx, n, in, in_pitch, 4, out, out_pitch, 3, on_device, [&](int grid, const uint8_t* di, size_t ip, uint8_t* dout, size_t op) {
    g1_smul_kernel<<<grid, kBlock, 0, ctx->compute>>>(ctx->d_tables, n, di, ip, dout, op);
  });
}
int pbh_g1_add_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return planes_impl(ctx, n, in, in_pitch, 6, out, out_pitch, 3, on_device, [&](int grid, const uint8_t* di, size_t ip, uint8_t* dout, size_t op) {
    g1_add_kernel<<<grid, kBlock, 0, ctx->compute>>>(ctx->d_tables, n, di, ip, dout, op);
  });
}
int pbh_kzg_commit_batch(pbh_ctx* ctx, size_t n, const uint8_t* coeffs, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return planes_impl(ctx, n, coeffs, in_pitch, 7, out, out_pitch, 3, on_device, [&](int grid, const uint8_t* di, size_t ip, uint8_t* dout, size_t op) {
    if (ctx->algo == PBH_ALGO_TABLE) {
      // four items per word when the layout allows and no coefficient can index past the SRS; the tail goes byte-wise
      const bool vec_ok = ctx->hs.K.n_pts >= 7 && ((uintptr_t)di % 4 == 0) && ((uintptr_t)dout % 4 == 0) && (ip % 4 == 0) && (op % 4 == 0);
      const size_t n4 = vec_ok ? n / 4 : 0;
      if (n4) {
        kzg_commit_table_vec_kernel<<<grid_for(ctx, n4, 8), kBlock, 0, ctx->compute>>>(ctx->hs.K, ctx->d_tables, n4, di, ip, dout, op);
        ctx->launches++;
      }
      if (n4 * 4 < n)
        kzg_commit_kernel<ALGO_TABLE><<<1, kBlock, 0, ctx->compute>>>(ctx->hs.K, ctx->d_tables, n - n4 * 4, di + n4 * 4, ip, dout + n4 * 4, op);
      else ctx->launches--;   // planes_impl counts one launch
    } else kzg_commit_kernel<ALGO_ARITH><<<grid, kBlock, 0, ctx->compute>>>(ctx->hs.K, ctx->d_tables, n, di, ip, dout, op);
  });
}
int pbh_pairing_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return planes_impl(ctx, n, in, in_pitch, 5, out, out_pitch, 2, on_device, [&](int grid, const uint8_t* di, size_t ip, uint8_t* dout, size_t op) {
    pairing_kernel<<<grid, kBlock, 0, ctx->compute>>>(ctx->d_tables, n, di, ip, dout, op);
  });
}

int pbh_gt_mul_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return planes_impl(ctx, n, in, in_pitch, 4, out, out_pitch, 2, on_device, [&](int grid, const uint8_t* di, size_t ip, uint8_t* dout, size_t op) {
    gt_kernel<0><<<grid, kBlock, 0, ctx->compute>>>(ctx->d_tables, n, di, ip, dout, op);
  });
}
int pbh_gt_pow600_batch(pbh_ctx* ctx, size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  return planes_impl(ctx, n, in, in_pitch, 2, out, out_pitch, 2, on_device, [&](int grid, const uint8_t* di, size_t ip, uint8_t* dout, size_t op) {
    gt_kernel<1><<<grid, kBlock, 0, ctx->compute>>>(ctx->d_tables, n, di, ip, dout, op);
  });
}

int pbh_poly_divrem_batch(pbh_ctx* ctx, size_t n, uint32_t ln, uint32_t ld, const uint8_t* num, size_t num_pitch, const uint8_t* den,
                          size_t den_pitch, uint8_t* q, size_t q_pitch, uint8_t* r, size_t r_pitch, uint8_t* status, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!num || !den || !q || !r || !status || num_pitch < n || den_pitch < n || q_pitch < n || r_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (ln < 1 || ln > 32 || ld < 1 || ld > 16) return fail(ctx, PBH_ERR_UNSUPPORTED, "1 <= ln <= 32, 1 <= ld <= 16");
  const uint8_t *d_num = num, *d_den = den; uint8_t *d_q = q, *d_r = r, *d_st = status; size_t np = num_pitch, dp = den_pitch, qp = q_pitch, rp = r_pitch;
  if (!on_device) {
    d_num = stg.in(num, num_pitch, n, ln, ce); CUDA_TRY(ctx, ce);
    d_den = stg.in(den, den_pitch, n, ld, ce); CUDA_TRY(ctx, ce);
    d_q = stg.in<uint8_t>(nullptr, 0, n, ln, ce); CUDA_TRY(ctx, ce);
    d_r = stg.in<uint8_t>(nullptr, 0, n, ld, ce); CUDA_TRY(ctx, ce);
    d_st = stg.in<uint8_t>(nullptr, 0, n, 1, ce); CUDA_TRY(ctx, ce);
    np = dp = qp = rp = n;
  }
  poly_divrem_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(ctx->d_tables, n, ln, ld, d_num, np, d_den, dp, d_q, qp, d_r, rp, d_st);
  SWEEP_FINISH(ctx);
  if (!on_device) {
    CUDA_TRY(ctx, stg.out(q, q_pitch, d_q, n, ln));
    CUDA_TRY(ctx, stg.out(r, r_pitch, d_r, n, ld));
    CUDA_TRY(ctx, stg.out(status, n, d_st, n, 1));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute));
  }
  return PBH_OK;
}

int pbh_poly_addsub_ragged_batch(pbh_ctx* ctx, size_t n, uint32_t la, uint32_t lb, int subtract, const uint8_t* a, size_t a_pitch,
                                 const uint8_t* b, size_t b_pitch, uint8_t* out, size_t out_pitch, int on_device) {
  SWEEP_PROLOGUE(ctx, n);
  if (!a || !b || !out || a_pitch < n || b_pitch < n || out_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  if (la < 1 || la > 64 || lb < 1 || lb > 64) return fail(ctx, PBH_ERR_UNSUPPORTED, "1 <= la, lb <= 64");
  const uint32_t lo = std::max(la, lb);
  const uint8_t *d_a = a, *d_b = b; uint8_t* d_out = out; size_t ap = a_pitch, bp = b_pitch, op = out_pitch;
  if (!on_device) {
    d_a = stg.in(a, a_pitch, n, la, ce); CUDA_TRY(ctx, ce);
    d_b = stg.in(b, b_pitch, n, lb, ce); CUDA_TRY(ctx, ce);
    d_out = stg.in<uint8_t>(nullptr, 0, n, lo, ce); CUDA_TRY(ctx, ce);
    ap = bp = op = n;
  }
  poly_addsub_ragged_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(n, la, lb, subtract, d_a, ap, d_b, bp, d_out, op);
  SWEEP_FINISH(ctx);
  if (!on_device) { CUDA_TRY(ctx, stg.out(out, out_pitch, d_out, n, lo)); CUDA_TRY(ctx, cudaStreamSynchronize(ctx->compute)); }
  return PBH_OK;
}

// ---- shard summaries, synthetic inputs, measurement --------------------------------------------------------
int pbh_pack_verdicts_dev(pbh_ctx* ctx, size_t n, const uint8_t* result, uint8_t* bitmap) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!result || !bitmap) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  pack_verdicts_kernel<<<grid_for(ctx, (n + 7) / 8, 8), kBlock, 0, ctx->compute>>>(n, result, bitmap);
  SWEEP_FINISH(ctx);
  return PBH_OK;
}

int pbh_digest_dev(pbh_ctx* ctx, size_t n, uint64_t first_index, uint32_t planes, const uint8_t* data, size_t pitch, uint64_t* out) {
  CTX_CHECK(ctx);
  if (!out) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaMemsetAsync(out, 0, sizeof(uint64_t), ctx->compute));
  if (n == 0) return PBH_OK;
  if (!data || pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad pointer or pitch");
  return launch_digest(ctx, ctx->compute, n, first_index, planes, data, pitch, out);
}

// Whether some row of the generator's witness table (x^2 + y^2 = z^2, laid out as generate_kernel lays it out) satisfies the
// context's gates and copy constraints.  Without one every full-path attempt ends in PBH_ST_UNSATISFIED.
static bool fullpath_satisfiable(const Consts& K) {
  for (uint32_t x = 0; x < 17; x++)
    for (uint32_t y = 0; y < 17; y++)
      for (uint32_t z = 0; z < 17; z++) {
        if ((x * x + y * y) % 17 != (z * z) % 17) continue;
        const uint32_t xx = x * x % 17, yy = y * y % 17, zz = z * z % 17;
        const uint32_t w[12] = {x, y, z, xx, x, y, z, yy, xx, yy, zz, zz};
        if (!unsatisfied(w, K)) return true;
      }
  return false;
}

int pbh_generate_inputs_dev(pbh_ctx* ctx, size_t n, uint64_t first_index, uint64_t seed, int dist, uint8_t* wit, size_t wit_pitch,
                            uint8_t* rnd, size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u, uint8_t* attempt) {
  CTX_CHECK(ctx);
  if (n == 0) return PBH_OK;
  if (!wit || !rnd || !chal || !u) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "null pointer");
  if (wit_pitch < n || rand_pitch < n || chal_pitch < n) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "pitch < n");
  if (dist != PBH_DIST_UNIFORM && dist != PBH_DIST_FULLPATH) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "unknown distribution");
  if (dist == PBH_DIST_FULLPATH && !fullpath_satisfiable(ctx->hs.K))
    return fail(ctx, PBH_ERR_UNSUPPORTED, "no witness of the generator's table satisfies this circuit: PBH_DIST_FULLPATH cannot succeed");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GenArgs A{n, first_index, seed, dist, wit, wit_pitch, rnd, rand_pitch, chal, chal_pitch, u, attempt, ctx->d_wtab};
  generate_kernel<<<grid_for(ctx, n, 8), kBlock, 0, ctx->compute>>>(ctx->hs.K, ctx->d_tables, A);
  SWEEP_FINISH(ctx);
  return PBH_OK;
}

int pbh_measure_int32_peak(pbh_ctx* ctx, int which, double* lane_ops_per_second) {
  CTX_CHECK(ctx);
  if (!lane_ops_per_second || which < 0 || which > 16) return fail(ctx, PBH_ERR_BAD_ARGUMENT, "bad argument");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  uint32_t* sink = nullptr;
  CUDA_TRY(ctx, cudaMalloc(&sink, 4));
  cudaEvent_t e0, e1;
  CUDA_TRY(ctx, cudaEventCreate(&e0));
  CUDA_TRY(ctx, cudaEventCreate(&e1));
  const uint32_t iters = 4096;
  const int grid = ctx->sm_count * 8;
  auto launch = [&]() {
    switch (which) {
      case 0: int32_peak_kernel<0><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 1: int32_peak_kernel<1><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 2: int32_peak_kernel<2><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 3: int32_peak_kernel<3><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 4: int32_peak_kernel<4><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 5: int32_peak_kernel<5><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 6: int32_peak_kernel<6><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 7: int32_peak_kernel<7><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 8: mac3_peak_kernel<0><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 9: mac3_peak_kernel<1><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 10: ffma2_peak_kernel<0><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 11: ffma2_peak_kernel<1><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 12: shift_peak_kernel<0><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 13: shift_peak_kernel<1><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 14: shift_peak_kernel<2><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      case 15: shift_peak_kernel<3><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
      default: shift_peak_kernel<4><<<grid, kBlock, 0, ctx->compute>>>(iters, 12345u, sink); break;
    }
    ctx->launches++;
  };
  for (int w = 0; w < 3; w++) launch();
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0, ctx->compute);
    launch();
    cudaEventRecord(e1, ctx->compute);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    // per inner repetition over the 8 chains: 8 ops (IMAD / FFMA / HFMA2 / dp4a / mixed), 16 for LOP3+IADD3,
    // 4 IMAD + 8 ALU for the mix, 16 for IMAD.HI + IADD
    const double per_rep = (which == 1 || which == 6) ? 16.0 : (which == 2 ? 12.0 : 8.0);
    double ops = (double)iters * 8.0 * per_rep * (double)grid * kBlock;
    if (ms > 0) best = std::max(best, ops / (ms * 1e-3));
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  CUDA_TRY(ctx, cudaGetLastError());
  *lane_ops_per_second = best;
  return PBH_OK;
}
