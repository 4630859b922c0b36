// Host side of the tcgen05 GEMM: TMA tensor-map encoding (driver entry point resolved at run time, so the
// library links against cudart only), the stream-K schedule and the persistent launch.
#pragma once
#include <cstdio>
#include <cstring>
#include <atomic>
#include <mutex>
#include <vector>

#include "gemm_sm100.cuh"

namespace td {

// ---- error plumbing shared by the whole library (C-ABI returns codes, td_last_error() returns this text)
inline char* last_error_buf() {
  static thread_local char buf[512] = "";
  return buf;
}
#define TD_FAIL(code, ...)                                        \
  do {                                                            \
    snprintf(td::last_error_buf(), 512, __VA_ARGS__);             \
    return (code);                                                \
  } while (0)
#define TD_CUDA(expr)                                                                             \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) TD_FAIL(-100 - int(_e), "%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

enum : int { TD_OK = 0, TD_ERR_ARG = -1, TD_ERR_UNSUPPORTED = -2, TD_ERR_DRIVER = -3 };

// ---- optional per-launch timing: when enabled (td_profile_enable) every kernel launch of the library is bracketed
// by a pair of CUDA events on the launch stream; td_profile_report() sums them per tag, td_profile_timeline() lists them
// with their offsets from the first record (events of different streams share the device clock, so this is a per-stream
// timeline). Off by default (zero cost). Launches may come from several host threads (autograd runs backward on its own).
// An event recorded between two kernels ends programmatic dependent launch there: with profiling on, every kernel starts after
// its predecessor has completed, so the per-kernel times include the prologue that PDL otherwise hides under the previous kernel.
struct ProfRecord { const char* tag; cudaEvent_t e0, e1; double work; cudaStream_t stream; };
struct Profiler {
  std::atomic<bool> on{false};
  std::mutex mu;
  std::vector<ProfRecord> recs;
  static Profiler& get() { static Profiler p; return p; }
};
struct ProfScope {
  cudaStream_t st; cudaEvent_t e1 = nullptr;
  // `work` = algorithmic FLOPs (GEMMs) or bytes (row kernels) of this launch, for the roofline report
  ProfScope(const char* tag, double work, cudaStream_t s) : st(s) {
    Profiler& p = Profiler::get();
    if (!p.on.load(std::memory_order_relaxed)) return;
    ProfRecord r{tag, nullptr, nullptr, work, s};
    cudaEventCreate(&r.e0); cudaEventCreate(&r.e1);
    cudaEventRecord(r.e0, st);
    e1 = r.e1;
    std::lock_guard<std::mutex> lock(p.mu);
    p.recs.push_back(r);
  }
  ~ProfScope() { if (e1) cudaEventRecord(e1, st); }
};

// ---- per-device state. Everything the library caches is keyed by the CUDA device that is current at the call, so one
// process may drive several GPUs.
constexpr int kMaxDevices = 32;
struct DeviceState {
  std::mutex mu;
  int sms = 0;
  int cc_major = -1;
  int* sk_flags = nullptr;  // pool of zeroed stream-K flag blocks, one block per launch, re-armed by the kernels
  std::atomic<unsigned> sk_seq{0};
  int* sched = nullptr;     // pool of {next unit, workers out of units, workers torn down, -} counters for the dynamic tile scheduler
  std::atomic<unsigned> sched_seq{0};
};
constexpr unsigned kSchedPairs = 1024;                       // a pair is re-armed (zeroed) by the kernel that used it
constexpr unsigned kSkFlagSlots = 256;                       // far more launches than can be in flight at once
constexpr int kSkFlagsPerSlot = 148 * kEpiWarps;             // [workers][CTAS][8] with workers * CTAS <= 148

inline int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return -1; }
  return dev;
}
inline DeviceState* device_state() {
  static DeviceState states[kMaxDevices];
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices) return nullptr;
  DeviceState& s = states[dev];
  if (s.cc_major < 0) {
    std::lock_guard<std::mutex> lock(s.mu);
    if (s.cc_major < 0) {
      int sms = 0, major = 0;
      if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
          cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
      s.sms = sms;
      s.cc_major = major;
    }
  }
  return &s;
}
inline int device_sm_count() {
  DeviceState* s = device_state();
  return (s && s->sms > 0) ? s->sms : 148;  // no device visible (size queries on a build box): assume a full B200
}
inline int* next_sk_flags() {
  DeviceState* s = device_state();
  if (!s) return nullptr;
  if (!s->sk_flags) {
    std::lock_guard<std::mutex> lock(s->mu);
    if (!s->sk_flags) {
      int* p = nullptr;
      const size_t bytes = sizeof(int) * (size_t)kSkFlagSlots * kSkFlagsPerSlot;
      if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
      if (cudaMemset(p, 0, bytes) != cudaSuccess) return nullptr;
      s->sk_flags = p;
    }
  }
  return s->sk_flags + (size_t)(s->sk_seq.fetch_add(1) % kSkFlagSlots) * kSkFlagsPerSlot;
}

// Every launch takes the next counter pair; no per-launch memset is needed.
inline int* next_sched_counter() {
  DeviceState* s = device_state();
  if (!s) return nullptr;
  if (!s->sched) {
    std::lock_guard<std::mutex> lock(s->mu);
    if (!s->sched) {
      int* p = nullptr;
      if (cudaMalloc(&p, sizeof(int) * 4 * kSchedPairs) != cudaSuccess) return nullptr;
      if (cudaMemset(p, 0, sizeof(int) * 4 * kSchedPairs) != cudaSuccess) return nullptr;
      s->sched = p;
    }
  }
  return s->sched + 4 * (s->sched_seq.fetch_add(1) % kSchedPairs);
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                        CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                        CUtensorMapFloatOOBfill);

inline PFN_tmapEncodeTiled tmap_encoder() {
  static PFN_tmapEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  });
  return fn;
}

inline int encode_2d(CUtensorMap* map, CUtensorMapDataType dt, const void* ptr, cuuint64_t dim0, cuuint64_t dim1,
                     cuuint64_t stride1_bytes, cuuint32_t box0, cuuint32_t box1, CUtensorMapSwizzle sw,
                     CUtensorMapL2promotion promo) {
  PFN_tmapEncodeTiled enc = tmap_encoder();
  if (!enc) TD_FAIL(TD_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || stride1_bytes % 16)
    TD_FAIL(TD_ERR_ARG, "TMA tensor needs a 16-byte aligned base and row pitch (ptr=%p pitch=%llu)", ptr, (unsigned long long)stride1_bytes);
  cuuint64_t gdim[2] = {dim0, dim1}, gstride[1] = {stride1_bytes};
  cuuint32_t box[2] = {box0, box1}, estr[2] = {1, 1};
  CUresult r = enc(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, promo,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_ERROR_INVALID_CONTEXT) {
    // a host thread that has not touched the runtime yet (e.g. autograd's backward thread) has no context bound: bind the
    // primary context of the current device and try again
    cudaFree(nullptr);
    r = enc(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, promo,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS)
    TD_FAIL(TD_ERR_DRIVER, "cuTensorMapEncodeTiled failed with CUresult %d (ptr=%p dims=%llu x %llu pitch=%llu box=%u x %u)", int(r), ptr,
            (unsigned long long)dim0, (unsigned long long)dim1, (unsigned long long)stride1_bytes, box0, box1);
  return TD_OK;
}

// bf16 operand with `rows` logical rows and contraction length K.
//   K-major : memory is [rows, K] (ld = elements between rows);  box = 64 (K) x box_rows
//   MN-major: memory is [K, rows] (ld = elements between k-rows); box = 64 (rows) x 64 (K)
inline int make_operand_map(CUtensorMap* map, const void* ptr, long long rows, long long K, long long ld,
                            bool mn_major, int box_rows) {
  if (!mn_major)
    return encode_2d(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, ptr, (cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)ld * 2, kBlockK,
                     (cuuint32_t)box_rows, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  return encode_2d(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, ptr, (cuuint64_t)rows, (cuuint64_t)K, (cuuint64_t)ld * 2, 64, kBlockK,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}
// Epilogue tensors [rows, cols] row-major, moved as 32-row x 32-column boxes: bf16 (64-byte box rows, 64-byte swizzle) or
// fp32 (128-byte box rows, 128-byte swizzle). Matches box64_off / box128_off in gemm_sm100.cuh.
inline int make_epilogue_map(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld, bool f32) {
  if (f32)
    return encode_2d(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, ptr, (cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)ld * 4, 32, 32,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE);
  return encode_2d(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, ptr, (cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)ld * 2, 32, 32,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE);
}

struct GemmOperand {
  const void* ptr;
  long long ld;   // elements
  bool mn_major;
};

// Workspace for the stream-K tail of one GEMM launch: one accumulator slot per CTA.
inline size_t gemm_sk_workspace_bytes() { return sizeof(float) * (size_t)device_sm_count() * kSkSlotFloats; }

// Largest number of tail ranges that share one tail tile when the R * KB tail k-blocks are cut into p.tail_workers ranges.
inline int max_tail_participants(const GemmParams& p, int R) {
  const int KB = p.num_k_blocks;
  int most = 1;
  for (int t = 0; t < R; ++t) {
    const int n = sk_worker_of(p, (t + 1) * KB - 1) - sk_worker_of(p, t * KB) + 1;
    if (n > most) most = n;
  }
  return most;
}

// Fill the schedule fields of `p` for `workers` workers. With a stream-K workspace the tiles left over after the full waves are
// cut along K into equal ranges (never shorter than kMinTailKBlocks); without one they form a last, partially filled wave.
// The number of ranges minimises the tail's estimated time in k-blocks: the longest range plus kTailFoldKBlocks for every
// partial the busiest owner folds in. More ranges shorten the MMA part but give each tail tile more contributors, and an
// owner folds those in one after another.
inline void plan_schedule(GemmParams& p, int max_workers, bool stream_k) {
  const int tiles = p.num_m_blocks * p.num_n_blocks;
  const int KB = p.num_k_blocks;
  int W = max_workers;
  if (tiles < W) {
    long long by_k = (long long)tiles * KB / kMinTailKBlocks;
    long long w = stream_k ? (by_k > tiles ? by_k : tiles) : tiles;
    W = int(w < max_workers ? w : max_workers);
    if (W < 1) W = 1;
  }
  p.workers = W;
  p.full_waves = tiles / W;
  const int R = tiles - p.full_waves * W;
  p.tail_workers = 0; p.tail_q = 0; p.tail_r = 0;
  if (stream_k && R > 0) {
    const long long units = (long long)R * KB;
    long long hi = units / kMinTailKBlocks;
    if (hi < R) hi = R;  // at least one worker per tile: a range never spans more than two tiles
    if (hi > W) hi = W;
    long long best_cost = -1;
    int best = int(hi);
    for (int wt = int(hi); wt >= R; --wt) {  // ties keep the larger count (the shorter ranges)
      p.tail_q = int(units / wt);
      p.tail_r = int(units % wt);
      const long long cost = (units + wt - 1) / wt + (long long)kTailFoldKBlocks * (max_tail_participants(p, R) - 1);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = wt; }
    }
    p.tail_workers = best;
    p.tail_q = int(units / best);
    p.tail_r = int(units % best);
    if (p.full_waves == 0) p.workers = best;  // every worker holds one tail range: launch no idle ones
  }
}

// `ws` (optional, gemm_sk_workspace_bytes()) enables the stream-K tail.
template <int CTAS, bool A_MN, bool B_MN, int EPI>
int launch_gemm(GemmOperand a, GemmOperand b, GemmParams p, void* ws, cudaStream_t stream, const char* tag = "gemm") {
  using S = GemmSmem<CTAS, EPI>;
  if (p.M <= 0 || p.N <= 0) return TD_OK;
  if (p.N % 32) TD_FAIL(TD_ERR_UNSUPPORTED, "GEMM N=%d must be a multiple of 32", p.N);
  if (p.K <= 0) TD_FAIL(TD_ERR_ARG, "GEMM K=%d must be positive (caller zero-fills empty contractions)", p.K);
  CUtensorMap ma, mb, mo0, mo1, maux;
  ScatterMaps smaps;
  memset(&mo0, 0, sizeof(mo0)); memset(&mo1, 0, sizeof(mo1)); memset(&maux, 0, sizeof(maux)); memset(&smaps, 0, sizeof(smaps));
  int rc = make_operand_map(&ma, a.ptr, p.M, p.K, a.ld, A_MN, kBlockM);
  if (rc) return rc;
  rc = make_operand_map(&mb, b.ptr, p.N, p.K, b.ld, B_MN, kBlockN / CTAS);
  if (rc) return rc;
  if (EPI == EPI_GATED && p.N % 64)
    TD_FAIL(TD_ERR_UNSUPPORTED, "gated GEMM: N=%d must be a multiple of 64 (whole (a, b) pairs)", p.N);
  // EPI_DGATED's output and aux are the interleaved [M, 2N] pair buffers; EPI_GATED's out1 is the contiguous [M, N / 2] product
  const long long out_cols = EPI == EPI_DGATED ? 2ll * p.N : p.N;
  if (EPI != EPI_F32_SCATTER && p.out0 != nullptr) {
    rc = make_epilogue_map(&mo0, p.out0, p.M, out_cols, p.ld_out, EPI == EPI_F32);
    if (rc) return rc;
  }
  if (EPI == EPI_BIAS_GELU) {
    rc = make_epilogue_map(&mo1, p.out1, p.M, p.N, p.ld_out, false);
    if (rc) return rc;
  }
  if (EPI == EPI_GATED) {
    rc = make_epilogue_map(&mo1, p.out1, p.M, p.N / 2, p.N / 2, false);
    if (rc) return rc;
  }
  if (EPI == EPI_F32_SCATTER) {
    if (p.scatter_rows <= 0 || p.scatter_rows % 32 || p.M % p.scatter_rows || p.M / p.scatter_rows > kMaxPeers)
      TD_FAIL(TD_ERR_ARG, "row-scattered GEMM: %d rows per owner must be a multiple of 32 and divide M=%d into at most %d blocks", p.scatter_rows, p.M, kMaxPeers);
    for (int o = 0; o < p.M / p.scatter_rows; ++o) {
      rc = make_epilogue_map(&smaps.m[o], p.scatter_dst[o], p.scatter_rows, p.N, p.ld_out, true);
      if (rc) return rc;
    }
  }
  if (EPI == EPI_DGELU || EPI == EPI_RESIDUAL || EPI == EPI_DGATED) {
    rc = make_epilogue_map(&maux, p.aux0, p.M, out_cols, p.ld_out, false);
    if (rc) return rc;
  }
  p.num_m_blocks = (p.M + kBlockM * CTAS - 1) / (kBlockM * CTAS);
  p.num_n_blocks = (p.N + kBlockN - 1) / kBlockN;
  p.num_k_blocks = (p.K + kBlockK - 1) / kBlockK;
  plan_schedule(p, device_sm_count() / CTAS, ws != nullptr);
  p.sk_partials = static_cast<float*>(ws);
  p.sched_counter = next_sched_counter();
  if (!p.sched_counter) TD_FAIL(TD_ERR_DRIVER, "cannot allocate the tile-scheduler counters");
  p.sk_flags = nullptr;
  if (p.tail_workers > 0) {
    p.sk_flags = next_sk_flags();
    if (!p.sk_flags) TD_FAIL(TD_ERR_DRIVER, "cannot allocate the stream-K flag pool");
  }

  auto kern = gemm_bf16_kernel<CTAS, A_MN, B_MN, EPI>;
  static std::atomic<bool> attr_set[kMaxDevices];  // per template instantiation, per device
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices) TD_FAIL(TD_ERR_DRIVER, "no current CUDA device");
  if (!attr_set[dev].load(std::memory_order_acquire)) {
    TD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    attr_set[dev].store(true, std::memory_order_release);
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(p.workers * CTAS);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTAS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // programmatic dependent launch: the prologue (barriers, TMEM, cluster sync) overlaps the previous kernel's tail
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  ProfScope prof(tag, 2.0 * double(p.M) * double(p.N) * double(p.K), stream);
  TD_CUDA(cudaLaunchKernelEx(&cfg, kern, ma, mb, mo0, mo1, maux, smaps, p));
  return TD_OK;
}

}  // namespace td
