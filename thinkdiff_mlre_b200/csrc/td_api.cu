// C ABI of libthinkdiff_b200.so (declared in include/thinkdiff_b200.h): argument checking, workspace carving and
// kernel launches for the ThinkDiff aligner hot path on sm_100a. No torch types, no global mutable state beyond
// cached device attributes; every launch goes to the caller's stream.
#include "thinkdiff_b200.h"

#include "gemm_host.cuh"
#include "rowops_sm100.cuh"
#include "peer_sm100.cuh"
#include "attn_sm100.cuh"

#include <cmath>
#include <initializer_list>

using namespace td;

namespace {

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Carver {
  uint8_t* base;
  size_t off = 0;
  explicit Carver(void* p) : base(static_cast<uint8_t*>(p)) {}
  template <class T>
  T* take(size_t n) {
    T* r = reinterpret_cast<T*>(base + off);
    off = align_up(off + n * sizeof(T), 256);
    return r;
  }
};

int check_device() {
  DeviceState* d = device_state();
  if (!d) TD_FAIL(TD_ERR_UNSUPPORTED, "no usable CUDA device");
  if (d->cc_major != 10) TD_FAIL(TD_ERR_UNSUPPORTED, "libthinkdiff_b200 needs an sm_100 (B200) device; there is no fallback path");
  return TD_OK;
}
#define TD_DEVICE_OR_RETURN()      \
  do {                             \
    int _rc = check_device();      \
    if (_rc) return _rc;           \
  } while (0)

// The update kernels are meant to run on SMs that a persistent GEMM has configured for the maximum shared-memory carve-out:
// ask for the same split (they use no shared memory themselves), so the SM never has to drain to reconfigure.
template <class K>
inline void prefer_max_shared(K kernel) {
  static std::atomic<bool> done[kMaxDevices];
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices || done[dev].load(std::memory_order_acquire)) return;
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaGetLastError();
  done[dev].store(true, std::memory_order_release);
}

inline int grid_for_rows(long long rows, int rows_per_block, int blocks_per_sm) {
  const long long want = (rows + rows_per_block - 1) / rows_per_block;
  const long long cap = (long long)device_sm_count() * blocks_per_sm;
  return int(want < cap ? (want > 0 ? want : 1) : cap);
}

// Launch configuration with programmatic dependent launch, for the row kernels that sit between the GEMMs on the train step's
// compute stream (cu_seqlens, pack, norm_mse_bwd, loss_finish, finish). Each of them calls grid_dependency_wait() before it
// touches global memory, as the GEMM kernel does.
struct PdlConfig {
  cudaLaunchAttribute attr;
  cudaLaunchConfig_t cfg;
  PdlConfig(dim3 grid, dim3 block, cudaStream_t st) {
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.stream = st;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
  }
  PdlConfig(const PdlConfig&) = delete;  // cfg points at attr
};

// Grid of the norm-backward kernels: up to `ctas_per_sm` CTAs per SM (2 for the plain backward, 1 for the fused norm + MSE +
// norm-backward), each with one contiguous slab of rows, a multiple of the kNormBwdRows rows it walks at a time.
inline int norm_grid(long long M, int ctas_per_sm, int* rows_per_cta) {
  int ctas = device_sm_count() * ctas_per_sm;
  long long rpc = (M + ctas - 1) / ctas;
  rpc = (rpc + kNormBwdRows - 1) / kNormBwdRows * kNormBwdRows;
  if (rpc < kNormBwdRows) rpc = kNormBwdRows;
  *rows_per_cta = int(rpc);
  return int((M + rpc - 1) / rpc);
}

inline bool dims_ok(int Din, int D) { return Din > 0 && D > 0 && Din % 64 == 0 && D % 64 == 0 && D <= 8 * kNormBwdThreads; }

// A pointer argument of an entry point, by name, and what it must be: non-null and 16-byte aligned (the default), 16-byte aligned
// when given (an optional buffer), or only non-null.
enum PtrRule { kNonNullAligned, kOptionalAligned, kNonNull };
struct Arg {
  const char* name;
  const void* ptr;
  PtrRule rule = kNonNullAligned;
};

// Fails with the entry's name and the first offending argument; every null check comes before the alignment checks.
int check_pointers(const char* fn, std::initializer_list<Arg> args) {
  for (const Arg& a : args)
    if (a.rule != kOptionalAligned && !a.ptr) TD_FAIL(TD_ERR_ARG, "%s: null pointer (%s)", fn, a.name);
  for (const Arg& a : args)
    if (a.rule != kNonNull && (reinterpret_cast<uintptr_t>(a.ptr) & 15)) TD_FAIL(TD_ERR_ARG, "%s: %s must be 16-byte aligned", fn, a.name);
  return TD_OK;
}

// Zeroed GEMM parameters for an [M, N] output (row pitch N) over a K-long contraction, alpha = 1.
GemmParams gemm_params(int64_t M, int32_t N, int64_t K) {
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = int(M); p.N = N; p.K = int(K);
  p.ld_out = N; p.alpha = 1.f;
  return p;
}

// The pack entries: rows = total_rows (varlen) or B * L_max (padded), each row_bytes long, copied by pack_rows_kernel<PADDED>.
template <bool PADDED>
int pack_launch(const char* fn, std::initializer_list<Arg> ptrs, const void* src, const void* src2, const int64_t* src_row_start,
                const int32_t* cu, int32_t B, int64_t rows, int32_t L_max, int64_t row_bytes, void* dst, int64_t* mask,
                int64_t* src_row_out, cudaStream_t st) {
  if (B < 0 || rows < 0 || L_max < 0 || row_bytes <= 0 || row_bytes % 16)
    TD_FAIL(TD_ERR_ARG, "%s: row_bytes=%lld must be a positive multiple of 16", fn, (long long)row_bytes);
  if (rows == 0 || B == 0) return TD_OK;
  int rc = check_pointers(fn, ptrs);
  if (rc) return rc;
  ProfScope prof(PADDED ? "pack_padded" : "pack_varlen", 2.0 * double(rows) * double(row_bytes), st);
  PdlConfig l(grid_for_rows(rows, 8, 8), 256, st);
  TD_CUDA(cudaLaunchKernelEx(&l.cfg, pack_rows_kernel<PADDED>, static_cast<const uint4*>(src),
                             reinterpret_cast<const long long*>(src_row_start), cu, B, (long long)rows, L_max, int(row_bytes / 16),
                             static_cast<uint4*>(dst), reinterpret_cast<long long*>(mask),
                             reinterpret_cast<long long*>(src_row_out), static_cast<const uint4*>(src2)));
  return TD_OK;
}

}  // namespace

extern "C" {

const char* td_last_error(void) { return last_error_buf(); }
int32_t td_version(void) { return 100; }
int32_t td_device_check(void) { return check_device(); }

// ------------------------------------------------------------------------------------------------ profiling
int32_t td_profile_enable(int32_t on) {
  Profiler& p = Profiler::get();
  std::lock_guard<std::mutex> lock(p.mu);
  for (auto& r : p.recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  p.recs.clear();
  p.on.store(on != 0);
  return TD_OK;
}

// Writes "tag,launches,total_ms,total_work\n" lines (work = FLOPs for gemm_* tags, algorithmic bytes otherwise).
int32_t td_profile_report(char* buf, int32_t buflen) {
  Profiler& p = Profiler::get();
  std::lock_guard<std::mutex> lock(p.mu);
  struct Agg { const char* tag; int n; double ms, work; };
  std::vector<Agg> agg;
  for (auto& r : p.recs) {
    if (cudaEventSynchronize(r.e1) != cudaSuccess) TD_FAIL(TD_ERR_DRIVER, "td_profile_report: event sync failed");
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    size_t i = 0;
    for (; i < agg.size(); ++i) if (!strcmp(agg[i].tag, r.tag)) break;
    if (i == agg.size()) agg.push_back({r.tag, 0, 0.0, 0.0});
    agg[i].n++; agg[i].ms += ms; agg[i].work += r.work;
  }
  int off = 0;
  for (auto& a : agg) {
    int w = snprintf(buf + off, buflen > off ? buflen - off : 0, "%s,%d,%.6f,%.6e\n", a.tag, a.n, a.ms, a.work);
    if (w < 0 || off + w >= buflen) TD_FAIL(TD_ERR_ARG, "td_profile_report: buffer too small");
    off += w;
  }
  if (buflen > 0) buf[off < buflen ? off : buflen - 1] = 0;
  return TD_OK;
}

// Writes one "tag,stream,start_ms,end_ms\n" line per recorded launch, times relative to the first record: the events of
// different streams are stamped by the same device clock, so this is a per-stream timeline of the library's kernels.
int32_t td_profile_timeline(char* buf, int32_t buflen) {
  Profiler& p = Profiler::get();
  std::lock_guard<std::mutex> lock(p.mu);
  int off = 0;
  if (buflen > 0) buf[0] = 0;
  if (p.recs.empty()) return TD_OK;
  cudaEvent_t base = p.recs[0].e0;
  for (auto& r : p.recs) {
    if (cudaEventSynchronize(r.e1) != cudaSuccess) TD_FAIL(TD_ERR_DRIVER, "td_profile_timeline: event sync failed");
    float t0 = 0.f, t1 = 0.f;
    cudaEventElapsedTime(&t0, base, r.e0);
    cudaEventElapsedTime(&t1, base, r.e1);
    int w = snprintf(buf + off, buflen > off ? buflen - off : 0, "%s,%p,%.4f,%.4f\n", r.tag, (void*)r.stream, t0, t1);
    if (w < 0 || off + w >= buflen) TD_FAIL(TD_ERR_ARG, "td_profile_timeline: buffer too small");
    off += w;
  }
  return TD_OK;
}

// ------------------------------------------------------------------------------------------------ pack
int32_t td_cu_seqlens(const int32_t* lens, int32_t B, int32_t* cu, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (B < 0 || !cu || (B > 0 && !lens)) TD_FAIL(TD_ERR_ARG, "td_cu_seqlens: bad arguments");
  PdlConfig l(1, 1024, (cudaStream_t)stream);
  TD_CUDA(cudaLaunchKernelEx(&l.cfg, cu_seqlens_kernel, lens, B, cu));
  return TD_OK;
}

int32_t td_pack_varlen_indexed(const void* src, const int64_t* src_row_start, const int32_t* cu, int32_t B,
                               int64_t total_rows, int64_t row_bytes, void* dst, int64_t* src_row_out, td_stream_t stream);

int32_t td_pack_varlen(const void* src, const int64_t* src_row_start, const int32_t* cu, int32_t B, int64_t total_rows,
                       int64_t row_bytes, void* dst, td_stream_t stream) {
  return td_pack_varlen_indexed(src, src_row_start, cu, B, total_rows, row_bytes, dst, nullptr, stream);
}

int32_t td_pack_varlen_indexed(const void* src, const int64_t* src_row_start, const int32_t* cu, int32_t B,
                               int64_t total_rows, int64_t row_bytes, void* dst, int64_t* src_row_out, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  return pack_launch<false>("td_pack_varlen", {{"src", src}, {"src_row_start", src_row_start, kNonNull}, {"cu", cu, kNonNull}, {"dst", dst}},
                            src, nullptr, src_row_start, cu, B, total_rows, 0, row_bytes, dst, nullptr, src_row_out, (cudaStream_t)stream);
}

int32_t td_pack_varlen2(const void* src, const void* src2, const int64_t* src_row_start, const int32_t* cu, int32_t B,
                        int64_t total_rows, int64_t row_bytes, void* dst, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  return pack_launch<false>("td_pack_varlen2",
                            {{"src", src}, {"src2", src2}, {"src_row_start", src_row_start, kNonNull}, {"cu", cu, kNonNull}, {"dst", dst}},
                            src, src2, src_row_start, cu, B, total_rows, 0, row_bytes, dst, nullptr, nullptr, (cudaStream_t)stream);
}

int32_t td_pack_padded(const void* src, const int64_t* src_row_start, const int32_t* cu, int32_t B, int32_t L_max,
                       int64_t row_bytes, void* dst, int64_t* mask, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  return pack_launch<true>("td_pack_padded", {{"src", src, kOptionalAligned}, {"src_row_start", src_row_start, kNonNull}, {"cu", cu, kNonNull},
                           {"dst", dst}}, src, nullptr, src_row_start, cu, B, (int64_t)B * L_max, L_max, row_bytes, dst, mask, nullptr,
                           (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ casts
int32_t td_cast_f32_to_bf16(const float* src, void* dst, int64_t n, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (n < 0) TD_FAIL(TD_ERR_ARG, "td_cast_f32_to_bf16: n < 0");
  if (n == 0) return TD_OK;
  if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15)
    TD_FAIL(TD_ERR_ARG, "td_cast_f32_to_bf16: buffers must be 16-byte aligned");
  const int grid = grid_for_rows((n + 7) / 8, 256, 8);
  {
    ProfScope prof("cast_f32_to_bf16", 6.0 * double(n), (cudaStream_t)stream);
    cast_f32_to_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, static_cast<__nv_bfloat16*>(dst), n);
  }
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

// ------------------------------------------------------------------------------------------------ norm
// y (bf16 or fp32) = x * rstd * g. With `ssq_part`, each row's sum of squares comes from the `nparts` partials the GEMM that wrote
// x left behind instead of from x itself. A null tag launches unprofiled.
static int rmsnorm_fwd_launch(const void* x, const float* ssq_part, int nparts, const float* g, float eps, int64_t M, int32_t D,
                              void* y, int32_t y_dtype, float* rstd, const char* tag, cudaStream_t st) {
  const int grid = grid_for_rows(M, 8, 8);
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  {
    ProfScope prof(tag, double(M) * D * (y_dtype == TD_DTYPE_BF16 ? 4.0 : 6.0), st);
    if (y_dtype == TD_DTYPE_BF16)
      rmsnorm_fwd_kernel<true><<<grid, 256, 0, st>>>(xb, ssq_part, nparts, g, eps, int(M), D, y, rstd);
    else
      rmsnorm_fwd_kernel<false><<<grid, 256, 0, st>>>(xb, ssq_part, nparts, g, eps, int(M), D, y, rstd);
  }
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_rmsnorm_fwd(const void* x, const float* g, float eps, int64_t M, int32_t D, void* y, int32_t y_dtype,
                       float* rstd, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (M < 0 || D <= 0 || D % 8 || D > 8 * 32 * kNormFwdMaxVec)
    TD_FAIL(TD_ERR_ARG, "td_rmsnorm_fwd: D=%d must be a positive multiple of 8, at most %d", D, 8 * 32 * kNormFwdMaxVec);
  if (M == 0) return TD_OK;
  return rmsnorm_fwd_launch(x, nullptr, 0, g, eps, M, D, y, y_dtype, rstd, nullptr, (cudaStream_t)stream);
}

int64_t td_rmsnorm_bwd_workspace_bytes(int64_t M, int32_t D) {
  int rpc;
  const int grid = norm_grid(M > 0 ? M : 1, 2, &rpc);
  return (int64_t)(2 * align_up(sizeof(float) * (size_t)grid * D, 256));
}

static int rmsnorm_bwd_impl(const void* dy, int32_t dy_dtype, const __nv_bfloat16* x, const float* rstd, const float* g,
                            int64_t M, int32_t D, __nv_bfloat16* dx, float* dg, float* dxsum, float scale, void* ws,
                            cudaStream_t st) {
  int rpc;
  const int grid = norm_grid(M, 2, &rpc);
  Carver c(ws);
  float* dg_part = c.take<float>((size_t)grid * D);
  float* db_part = c.take<float>((size_t)grid * D);
  {
  ProfScope prof("rmsnorm_bwd", double(M) * D * (dy_dtype == TD_DTYPE_BF16 ? 6.0 : 8.0), st);
  if (dy_dtype == TD_DTYPE_BF16)
    rmsnorm_bwd_kernel<true><<<grid, kNormBwdThreads, 0, st>>>(dy, x, rstd, g, int(M), D, rpc, dx, dg_part, db_part);
  else
    rmsnorm_bwd_kernel<false><<<grid, kNormBwdThreads, 0, st>>>(dy, x, rstd, g, int(M), D, rpc, dx, dg_part, db_part);
  }
  TD_CUDA(cudaGetLastError());
  if (dg || dxsum) {  // one column-sum job per requested output (grid.y)
    const bool both = dg && dxsum;
    colsum_finish_kernel<<<dim3((D + 31) / 32, both ? 2 : 1), 256, 0, st>>>(dg ? dg_part : db_part, dg ? dg : dxsum,
                                                                          both ? db_part : nullptr, both ? dxsum : nullptr, grid, D, scale);
  }
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_rmsnorm_bwd(const void* dy, int32_t dy_dtype, const void* x, const float* rstd, const float* g, int64_t M,
                       int32_t D, void* dx, float* dg, float* dxsum, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (M < 0 || D <= 0 || D % 8 || D > 8 * kNormBwdThreads)
    TD_FAIL(TD_ERR_UNSUPPORTED, "td_rmsnorm_bwd: D=%d must be a multiple of 8 and <= %d", D, 8 * kNormBwdThreads);
  if (M == 0) {
    if (dg) TD_CUDA(cudaMemsetAsync(dg, 0, sizeof(float) * D, (cudaStream_t)stream));
    if (dxsum) TD_CUDA(cudaMemsetAsync(dxsum, 0, sizeof(float) * D, (cudaStream_t)stream));
    return TD_OK;
  }
  if (ws_bytes < td_rmsnorm_bwd_workspace_bytes(M, D)) TD_FAIL(TD_ERR_ARG, "td_rmsnorm_bwd: workspace too small");
  return rmsnorm_bwd_impl(dy, dy_dtype, static_cast<const __nv_bfloat16*>(x), rstd, g, M, D,
                          static_cast<__nv_bfloat16*>(dx), dg, dxsum, 1.0f, ws, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ GEMM entries
int64_t td_gemm_workspace_bytes(void) { return (int64_t)align_up(gemm_sk_workspace_bytes(), 256); }

namespace {
// the stream-K workspace is optional at the test / utility entries: without it the leftover tiles run as a last partial wave
inline void* sk_ws_or_null(void* ws, int64_t ws_bytes) { return (ws && ws_bytes >= td_gemm_workspace_bytes()) ? ws : nullptr; }

// The GEMM shapes the entries share. `a` [M, K] is K-major throughout; `sk` is the optional stream-K workspace.

// out [M, N] bf16 = bf16(a . w^T (+ bias)), w [N, K] K-major: a linear layer
int gemm_linear(const void* a, int64_t M, int32_t K, const void* w, int32_t N, const void* bias, void* out, void* sk, cudaStream_t st,
                const char* tag) {
  GemmParams p = gemm_params(M, N, K);
  p.out0 = out; p.bias = static_cast<const __nv_bfloat16*>(bias);
  return launch_gemm<2, false, false, EPI_BF16>({a, K, false}, {w, K, false}, p, sk, st, tag);
}

// out [M, N] = a . w, w [K, N] read MN-major in place (the input gradient of a linear layer): bf16, or fp32 when `f32`;
// `accumulate` (fp32 only): out += a . w by TMA reduce-add
int gemm_linear_dx(const void* a, int64_t M, int64_t K, const void* w, int32_t N, void* out, bool f32, void* sk, cudaStream_t st,
                   const char* tag, bool accumulate = false) {
  GemmParams p = gemm_params(M, N, K);
  p.out0 = out; p.accumulate = accumulate;
  if (f32) return launch_gemm<2, false, true, EPI_F32>({a, K, false}, {w, N, true}, p, sk, st, tag);
  return launch_gemm<2, false, true, EPI_BF16>({a, K, false}, {w, N, true}, p, sk, st, tag);
}

// out [M, N] bf16 = bf16(x + bf16(a . w^T)), w [N, K] K-major: the closing projection of a residual sublayer
int gemm_residual(const void* a, int64_t M, int32_t K, const void* w, int32_t N, const void* x, void* out, void* sk, cudaStream_t st,
                  const char* tag) {
  GemmParams p = gemm_params(M, N, K);
  p.out0 = out; p.aux0 = x;
  return launch_gemm<2, false, false, EPI_RESIDUAL>({a, K, false}, {w, K, false}, p, sk, st, tag);
}

// The aligner's Linear1: h0 = x . W1^T + b1 [M, D] and h1 = bf16(gelu(h0))
int gemm_fwd1(const void* x, int64_t M, int32_t Din, const void* W1, int32_t D, const void* b1, void* h0, void* h1, void* sk,
              cudaStream_t st) {
  GemmParams p = gemm_params(M, D, Din);
  p.out0 = h0; p.out1 = h1; p.bias = static_cast<const __nv_bfloat16*>(b1);
  return launch_gemm<2, false, false, EPI_BIAS_GELU>({x, Din, false}, {W1, Din, false}, p, sk, st, "gemm_fwd1_bias_gelu");
}

// The aligner's Linear2: h2 = bf16(h1 . W2^T + b2) [M, D], with per-row sum-of-squares partials in ssq_part for the norm after it
int gemm_fwd2(const void* h1, int64_t M, int32_t D, const void* W2, const void* b2, void* h2, float* ssq_part, void* sk,
              cudaStream_t st) {
  GemmParams p = gemm_params(M, D, D);
  p.out0 = h2; p.bias = static_cast<const __nv_bfloat16*>(b2); p.red0 = ssq_part;
  return launch_gemm<2, false, false, EPI_BIAS_SSQ>({h1, D, false}, {W2, D, false}, p, sk, st, "gemm_fwd2_bias_ssq");
}
}  // namespace

int32_t td_linear_bf16(const void* x, int64_t M, int32_t K, const void* W, int32_t N, const void* bias, void* out, void* ws,
                       int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (M < 0 || K <= 0 || N <= 0 || K % 8 || N % 32) TD_FAIL(TD_ERR_UNSUPPORTED, "td_linear_bf16: need K %% 8 == 0, N %% 32 == 0");
  if (M == 0) return TD_OK;
  return gemm_linear(x, M, K, W, N, bias, out, sk_ws_or_null(ws, ws_bytes), (cudaStream_t)stream, "gemm_linear");
}

int32_t td_linear_bf16_dx(const void* dy, int64_t M, int32_t N, const void* W, int32_t K, void* dx, void* ws, int64_t ws_bytes,
                          td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (M < 0 || K <= 0 || N <= 0 || N % 8 || K % 64) TD_FAIL(TD_ERR_UNSUPPORTED, "td_linear_bf16_dx: need N %% 8 == 0, K %% 64 == 0");
  if (M == 0) return TD_OK;
  // output [M, K]; the contraction runs over the N rows of W
  return gemm_linear_dx(dy, M, N, W, K, dx, false, sk_ws_or_null(ws, ws_bytes), (cudaStream_t)stream, "gemm_linear_dx");
}

int32_t td_gemm_bf16_f32out(const void* A, int64_t lda, int32_t a_mn, const void* B, int64_t ldb, int32_t b_mn, int64_t M,
                            int32_t N, int64_t K, float alpha, float* out, int32_t cta_pair, int32_t accumulate, void* ws,
                            int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (M <= 0 || N <= 0 || K <= 0) TD_FAIL(TD_ERR_ARG, "td_gemm_bf16_f32out: empty problem");
  GemmParams p = gemm_params(M, N, K);
  p.out0 = out; p.alpha = alpha; p.accumulate = accumulate != 0;
  cudaStream_t st = (cudaStream_t)stream;
  void* sk = sk_ws_or_null(ws, ws_bytes);
  GemmOperand a{A, lda, a_mn != 0}, b{B, ldb, b_mn != 0};
  const int sel = (cta_pair ? 4 : 0) | (a_mn ? 2 : 0) | (b_mn ? 1 : 0);
  switch (sel) {
    case 0: return launch_gemm<1, false, false, EPI_F32>(a, b, p, sk, st);
    case 1: return launch_gemm<1, false, true, EPI_F32>(a, b, p, sk, st);
    case 2: return launch_gemm<1, true, false, EPI_F32>(a, b, p, sk, st);
    case 3: return launch_gemm<1, true, true, EPI_F32>(a, b, p, sk, st);
    case 4: return launch_gemm<2, false, false, EPI_F32>(a, b, p, sk, st);
    case 5: return launch_gemm<2, false, true, EPI_F32>(a, b, p, sk, st);
    case 6: return launch_gemm<2, true, false, EPI_F32>(a, b, p, sk, st);
    default: return launch_gemm<2, true, true, EPI_F32>(a, b, p, sk, st);
  }
}

// ------------------------------------------------------------------------------------------------ aligner forward
namespace {
struct FwdWorkspace {
  float* ssq_part;
  void* sk;
  size_t bytes;
};
FwdWorkspace carve_fwd(void* ws, int64_t M, int32_t D) {
  Carver c(ws);
  FwdWorkspace w;
  const size_t nparts = 2 * ((size_t)(D + kBlockN - 1) / kBlockN);  // two column halves per N tile
  w.ssq_part = c.take<float>(nparts * (size_t)(M > 0 ? M : 1));
  w.sk = c.take<uint8_t>(gemm_sk_workspace_bytes());
  w.bytes = c.off;
  return w;
}
}  // namespace

int64_t td_aligner_fwd_workspace_bytes(int64_t M, int32_t Din, int32_t D) {
  (void)Din;
  return (int64_t)carve_fwd(nullptr, M, D).bytes;
}

int32_t td_aligner_fwd(const void* x, int64_t M, int32_t Din, int32_t D, const void* W1, const void* b1, const void* W2,
                       const void* b2, const float* g, float eps, void* h0, void* h1, void* h2, float* rstd, void* y,
                       int32_t y_dtype, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!dims_ok(Din, D)) TD_FAIL(TD_ERR_UNSUPPORTED, "td_aligner_fwd: Din=%d, D=%d must be multiples of 64 (D <= 4096)", Din, D);
  if (M < 0 || M > 0x7fffffffll / D) TD_FAIL(TD_ERR_ARG, "td_aligner_fwd: M=%lld out of range", (long long)M);
  if (M == 0) return TD_OK;
  if (!x || !W1 || !W2 || !g || !h1 || !h2 || !y) TD_FAIL(TD_ERR_ARG, "td_aligner_fwd: null pointer");
  if (ws_bytes < td_aligner_fwd_workspace_bytes(M, Din, D)) TD_FAIL(TD_ERR_ARG, "td_aligner_fwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  FwdWorkspace w = carve_fwd(ws, M, D);
  // sum-of-squares partials: one per 128-column half tile that exists (the last N tile may be half empty)
  const int nblk = (D + kEpiColsPerWarp - 1) / kEpiColsPerWarp;

  int rc = gemm_fwd1(x, M, Din, W1, D, b1, h0, h1, w.sk, st);
  if (rc) return rc;
  rc = gemm_fwd2(h1, M, D, W2, b2, h2, w.ssq_part, w.sk, st);
  if (rc) return rc;
  return rmsnorm_fwd_launch(h2, w.ssq_part, nblk, g, eps, M, D, y, y_dtype, rstd, "rmsnorm_fwd", st);
}

// ------------------------------------------------------------------------------------------------ aligner backward
namespace {
struct BwdWorkspace {
  __nv_bfloat16* dh2;
  __nv_bfloat16* dh0;
  void* norm_ws;
  float* db1_part;
  int db1_rows;
  void* sk;
  size_t bytes;
};
BwdWorkspace carve_bwd(void* ws, int64_t M, int32_t D) {
  Carver c(ws);
  BwdWorkspace w;
  const size_t m = (size_t)(M > 0 ? M : 1);
  w.dh2 = c.take<__nv_bfloat16>(m * D);
  w.dh0 = c.take<__nv_bfloat16>(m * D);
  w.norm_ws = c.take<uint8_t>((size_t)td_rmsnorm_bwd_workspace_bytes((int64_t)m, D));
  w.db1_rows = int((m + kBlockM - 1) / kBlockM + 1) * 4;  // one partial row per 32-row warp slab (+1 pair padding)
  w.db1_part = c.take<float>((size_t)w.db1_rows * D);
  w.sk = c.take<uint8_t>(gemm_sk_workspace_bytes());
  w.bytes = c.off;
  return w;
}

// The norm kernel of the fused path leaves [grid][D] dg partials, [grid][D] db2 partials and [grid] loss partials behind.
struct NormPartials {
  float* dg_part;
  float* db_part;
  float* loss_part;
  int grid, rows_per_cta;
  size_t bytes;
};
NormPartials carve_norm_partials(void* buf, int64_t M, int32_t D) {
  NormPartials n;
  n.grid = norm_grid(M > 0 ? M : 1, 1, &n.rows_per_cta);
  Carver c(buf);
  n.dg_part = c.take<float>((size_t)n.grid * D);
  n.db_part = c.take<float>((size_t)n.grid * D);
  n.loss_part = c.take<float>((size_t)n.grid);
  n.bytes = c.off;
  return n;
}

// Row-sharded destinations of the two weight gradients (data parallel over peer memory): dW?[o] = where the rows owned by
// rank o go (a [D / world, cols] fp32 block in rank o's memory, this rank's slot). world == 0: plain local outputs.
struct ScatterDst {
  int world = 0;
  int rank = -1;  // this rank (>= 0: owner-grouped raster rotated so that concurrent ranks store to different owners)
  // td_peer_fold: the protocol's tiny launches folded into this call's kernels
  int* signal[kMaxPeers] = {};   // counter bumped at every rank by the LAST weight-gradient GEMM of the call, at its end
  int n_signal = 0;
  float* post[kMaxPeers] = {};   // this rank's small-vector slot at every rank: the finisher stores db1 / dg / db2 there too
  int n_post = 0;
  const float* post_base = nullptr;
  long long post_numel = 0;
  float* dW1[kMaxPeers] = {};
  float* dW2[kMaxPeers] = {};
};

struct BwdExtras {
  float* stats = nullptr;   // inf-check counter (StepCtl)
  int accumulate = 0;       // add into the gradient buffers (micro-batch accumulation); local outputs only
  float* loss_out = nullptr;  // finish the fused path's deferred loss in the backward's finisher launch
  const NormPartials* np = nullptr;
  float loss_div = 1.f;
};

// Rows per owner and the NVLink traffic shaping of a row-scattered GEMM (see GemmParams::raster_group_m): tiles are grouped by
// owner, and rank r starts with the rows of owner r + 1 and ends with its own (local) rows. Only when an owner's rows are whole
// pair tiles (256 rows).
void set_scatter_raster(GemmParams& p, int world, int rank) {
  p.scatter_rows = p.M / world;
  const int tile_m = 2 * kBlockM;
  if (rank >= 0 && rank < world && world > 1 && p.scatter_rows % tile_m == 0) {
    const int per_owner = p.scatter_rows / tile_m;
    p.raster_group_m = per_owner < kGroupM ? per_owner : kGroupM;
    p.raster_rot_m = ((rank + 1) % world) * per_owner;
  }
}

int launch_dw_gemm(GemmOperand a, GemmOperand b, GemmParams& p, float* const* dst, int world, int rank, void* sk, cudaStream_t st,
                   const char* tag, const ScatterDst* signal_from = nullptr) {
  if (world <= 0) return launch_gemm<2, true, true, EPI_F32>(a, b, p, sk, st, tag);
  if (signal_from != nullptr) {
    for (int o = 0; o < signal_from->n_signal; ++o) p.post_signal[o] = signal_from->signal[o];
    p.post_signal_n = signal_from->n_signal;
  }
  if (p.M % world || (p.M / world) % 32) TD_FAIL(TD_ERR_UNSUPPORTED, "row-scattered GEMM: %d rows over %d ranks must give a multiple of 32 rows per rank", p.M, world);
  for (int o = 0; o < world; ++o) p.scatter_dst[o] = dst[o];
  set_scatter_raster(p, world, rank);
  return launch_gemm<2, true, true, EPI_F32_SCATTER>(a, b, p, sk, st, tag);
}

// Backward from dh2 (already in the workspace or caller-provided), in this order: dh0 GEMM (+ db1 partials) -> finisher
// (db1 | dg, db2 | loss, whichever the phases ask for, ONE launch) -> dW1 GEMM -> dW2 GEMM.
int bwd_from_dh2(const __nv_bfloat16* dh2, const void* x, const void* h0, const void* h1, const void* W2, int64_t M,
                 int32_t Din, int32_t D, float scale, const float* scale_ptr, float* dW1, float* db1, float* dW2, float* db2,
                 float* dg, BwdWorkspace& w, int32_t phases, cudaStream_t st, const ScatterDst* sc, const BwdExtras& ex) {
  const int world = sc ? sc->world : 0;
  const bool do_gelu = (phases & (TD_BWD_PHASE_GELU_W1 | TD_BWD_PHASE_GELU_ONLY)) != 0;
  const bool do_small2 = ex.np != nullptr && (phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_SMALL2_ONLY)) != 0;
  if (do_gelu) {
    // dh0 = bf16( bf16(scale_ptr * dh2 . W2) * gelu'(h0) ), plus per-slab column sums for db1
    GemmParams p = gemm_params(M, D, D);
    p.alpha_ptr = scale_ptr;
    p.out0 = w.dh0; p.aux0 = h0; p.red0 = w.db1_part;
    int rc = launch_gemm<2, false, true, EPI_DGELU>({dh2, D, false}, {W2, D, true}, p, w.sk, st, "gemm_dh0_dgelu");
    if (rc) return rc;
  }
  if (do_gelu || do_small2 || ex.loss_out != nullptr) {
    FinishParams f;
    memset(&f, 0, sizeof(f));
    f.N = D; f.scale = scale; f.accumulate = ex.accumulate; f.stats = ex.stats;
    f.scale_ptr = scale_ptr;
    if (do_small2) {
      // dg / db2 = (grad_scale * upstream) * column sums of the partials the fused forward pass left behind
      f.job[f.njobs++] = FinishJob{ex.np->dg_part, dg, ex.np->grid, 1};
      f.job[f.njobs++] = FinishJob{ex.np->db_part, db2, ex.np->grid, 1};
    }
    if (do_gelu) {
      // db1's partials already carry the upstream scalar (the dh0 GEMM applied it to dh1)
      const int slabs = int((M + 2 * kBlockM - 1) / (2 * kBlockM)) * 2 * 4;  // pair tiles: 2 slabs x 4 warps each
      f.job[f.njobs++] = FinishJob{w.db1_part, db1, slabs, 0};
    }
    if (ex.loss_out != nullptr && ex.np != nullptr) {
      f.loss_part = ex.np->loss_part; f.loss_P = ex.np->grid; f.loss_out = ex.loss_out; f.loss_div = ex.loss_div;
    }
    if (sc != nullptr && sc->n_post > 0) {
      for (int o = 0; o < sc->n_post; ++o) f.post[o] = sc->post[o];
      f.n_post = sc->n_post; f.post_base = sc->post_base; f.post_numel = sc->post_numel;
    }
    if (f.njobs > 0 || f.loss_out != nullptr) {
      PdlConfig l(dim3((D + 31) / 32, f.njobs + (f.loss_out ? 1 : 0)), 256, st);
      TD_CUDA(cudaLaunchKernelEx(&l.cfg, finish_kernel, f));
    }
  }
  if (phases & (TD_BWD_PHASE_GELU_W1 | TD_BWD_PHASE_W1_ONLY)) {
    // dW1[D, Din] = scale * dh0^T . x   (dh0 already carries the upstream scalar; W1_ONLY: dh0 is in the workspace from a GELU_ONLY call)
    GemmParams p = gemm_params(D, Din, M);
    p.alpha = scale; p.out0 = dW1; p.stats = ex.stats; p.accumulate = ex.accumulate;
    const bool last = !(phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_W2_ONLY));  // the call's last GEMM carries the signal
    int rc = launch_dw_gemm({w.dh0, D, true}, {x, Din, true}, p, sc ? sc->dW1 : nullptr, world, sc ? sc->rank : -1, w.sk, st,
                            world ? "gemm_dW1_scatter" : "gemm_dW1", last ? sc : nullptr);
    if (rc) return rc;
  }
  if (phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_W2_ONLY)) {
    // dW2[D, D] = scale * dh2^T . h1  (contraction over tokens; both operands MN-major)
    GemmParams p = gemm_params(D, D, M);
    p.alpha = scale; p.alpha_ptr = scale_ptr; p.out0 = dW2; p.stats = ex.stats;
    p.accumulate = ex.accumulate;
    int rc = launch_dw_gemm({dh2, D, true}, {h1, D, true}, p, sc ? sc->dW2 : nullptr, world, sc ? sc->rank : -1, w.sk, st,
                            world ? "gemm_dW2_scatter" : "gemm_dW2", sc);
    if (rc) return rc;
  }
  return TD_OK;
}

int zero_grads(int32_t Din, int32_t D, float* dW1, float* db1, float* dW2, float* db2, float* dg, int32_t phases,
               cudaStream_t st) {
  if (phases & TD_BWD_PHASE_NORM_W2) {
    TD_CUDA(cudaMemsetAsync(dW2, 0, sizeof(float) * (size_t)D * D, st));
    TD_CUDA(cudaMemsetAsync(db2, 0, sizeof(float) * D, st));
    TD_CUDA(cudaMemsetAsync(dg, 0, sizeof(float) * D, st));
  }
  if (phases & TD_BWD_PHASE_GELU_W1) {
    TD_CUDA(cudaMemsetAsync(dW1, 0, sizeof(float) * (size_t)D * Din, st));
    TD_CUDA(cudaMemsetAsync(db1, 0, sizeof(float) * D, st));
  }
  return TD_OK;
}
}  // namespace

int64_t td_aligner_bwd_workspace_bytes(int64_t M, int32_t Din, int32_t D) {
  (void)Din;
  return (int64_t)carve_bwd(nullptr, M, D).bytes;
}

int32_t td_aligner_bwd(const void* dy, int32_t dy_dtype, const void* x, const void* h0, const void* h1, const void* h2,
                       const float* rstd, const void* W2, const float* g, int64_t M, int32_t Din, int32_t D,
                       float grad_scale, float* dW1, float* db1, float* dW2, float* db2, float* dg, void* ws,
                       int64_t ws_bytes, int32_t phases, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!dims_ok(Din, D)) TD_FAIL(TD_ERR_UNSUPPORTED, "td_aligner_bwd: Din=%d, D=%d must be multiples of 64 (D <= 4096)", Din, D);
  if (M < 0 || M > 0x7fffffffll / D) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd: M=%lld out of range", (long long)M);
  cudaStream_t st = (cudaStream_t)stream;
  if (M == 0) return zero_grads(Din, D, dW1, db1, dW2, db2, dg, phases, st);  // empty shard: exact zeros
  if (ws_bytes < td_aligner_bwd_workspace_bytes(M, Din, D)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd: workspace too small");
  BwdWorkspace w = carve_bwd(ws, M, D);
  if (phases & TD_BWD_PHASE_NORM_W2) {
    if (!dy || !h1 || !h2 || !rstd || !g || !dW2 || !db2 || !dg) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd: null pointer (phase 1)");
    // T5LayerNorm backward -> dh2 (bf16), dg, db2
    int rc = rmsnorm_bwd_impl(dy, dy_dtype, static_cast<const __nv_bfloat16*>(h2), rstd, g, M, D, w.dh2, dg, db2, grad_scale,
                              w.norm_ws, st);
    if (rc) return rc;
  }
  if ((phases & TD_BWD_PHASE_GELU_W1) && (!x || !h0 || !W2 || !dW1 || !db1)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd: null pointer (phase 2)");
  BwdExtras ex;  // (dg / db2 were finished by rmsnorm_bwd_impl: no norm partials here)
  return bwd_from_dh2(w.dh2, x, h0, h1, W2, M, Din, D, grad_scale, nullptr, dW1, db1, dW2, db2, dg, w, phases, st, nullptr, ex);
}

// ------------------------------------------------------------------------------------------------ fused aligner + MSE
int64_t td_aligner_mse_fwd_workspace_bytes(int64_t M, int32_t Din, int32_t D) {
  const size_t m = (size_t)(M > 0 ? M : 1);
  return td_aligner_fwd_workspace_bytes(M, Din, D) + (int64_t)align_up(sizeof(__nv_bfloat16) * m * D, 256) + 256;
}

int64_t td_aligner_norm_partials_bytes(int64_t M, int32_t D) { return (int64_t)carve_norm_partials(nullptr, M, D).bytes; }

int32_t td_aligner_mse_fwd(const void* x, int64_t M, int32_t Din, int32_t D, const void* W1, const void* b1,
                           const void* W2, const void* b2, const float* g, float eps, const void* target,
                           int32_t target_dtype, const int64_t* target_row_index, void* h0, void* h1, void* dh2,
                           void* norm_partials, float* loss, void* ws, int64_t ws_bytes, int32_t stages,
                           td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!dims_ok(Din, D)) TD_FAIL(TD_ERR_UNSUPPORTED, "td_aligner_mse_fwd: Din=%d, D=%d must be multiples of 64 (D <= 4096)", Din, D);
  if (M <= 0 || M > 0x7fffffffll / D) TD_FAIL(TD_ERR_ARG, "td_aligner_mse_fwd: M=%lld out of range (needs at least one token)", (long long)M);
  if (!x || !W1 || !W2 || !g || !target || !h0 || !h1 || !dh2 || !norm_partials)
    TD_FAIL(TD_ERR_ARG, "td_aligner_mse_fwd: null pointer");
  if (!(stages & TD_FWD_STAGE_DEFER_LOSS) && !loss) TD_FAIL(TD_ERR_ARG, "td_aligner_mse_fwd: loss pointer is null");
  if (ws_bytes < td_aligner_mse_fwd_workspace_bytes(M, Din, D)) TD_FAIL(TD_ERR_ARG, "td_aligner_mse_fwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  FwdWorkspace w = carve_fwd(ws, M, D);
  Carver c(static_cast<uint8_t*>(ws) + w.bytes);
  const int nparts = (D + kEpiColsPerWarp - 1) / kEpiColsPerWarp;
  __nv_bfloat16* h2 = c.take<__nv_bfloat16>((size_t)M * D);
  NormPartials np = carve_norm_partials(norm_partials, M, D);  // consumed by td_aligner_bwd_dh2

  int rc;
  if (stages & TD_FWD_STAGE_LINEAR1) {  // Linear1 + GELU (reads W1, b1 only)
    rc = gemm_fwd1(x, M, Din, W1, D, b1, h0, h1, w.sk, st);
    if (rc) return rc;
  }
  if (!(stages & TD_FWD_STAGE_REST)) return TD_OK;
  rc = gemm_fwd2(h1, M, D, W2, b2, h2, w.ssq_part, w.sk, st);
  if (rc) return rc;
  const float dy_coef = 2.0f / (float(M) * float(D));
  const long long* tri = reinterpret_cast<const long long*>(target_row_index);
  {
    ProfScope prof("norm_mse_bwd_fused", double(M) * D * (4.0 + (target_dtype == TD_DTYPE_BF16 ? 2.0 : 4.0)), st);
    PdlConfig l(np.grid, kNormBwdThreads, st);
    TD_CUDA(cudaLaunchKernelEx(&l.cfg, target_dtype == TD_DTYPE_BF16 ? norm_mse_bwd_kernel<true> : norm_mse_bwd_kernel<false>, h2,
                               w.ssq_part, nparts, eps, g, target, tri, int(M), D, np.rows_per_cta, dy_coef,
                               static_cast<__nv_bfloat16*>(dh2), np.dg_part, np.db_part, np.loss_part));
  }
  if (!(stages & TD_FWD_STAGE_DEFER_LOSS)) {
    PdlConfig l(1, 256, st);
    TD_CUDA(cudaLaunchKernelEx(&l.cfg, loss_finish_kernel, static_cast<const float*>(np.loss_part), np.grid,
                               static_cast<const float*>(nullptr), float(D), loss, float(M)));
  }
  return TD_OK;
}

}  // extern "C"
namespace {
int bwd_dh2_impl(const void* dh2, const void* x, const void* h0, const void* h1, const void* W2,
                 const void* norm_partials, int64_t M, int32_t Din, int32_t D,
                 float grad_scale, const float* grad_scale_ptr, float* dW1, float* db1, float* dW2, float* db2,
                 float* dg, float* loss_out, float* stats, int32_t accumulate, void* ws, int64_t ws_bytes, int32_t phases,
                 td_stream_t stream, const ScatterDst* sc) {
  TD_DEVICE_OR_RETURN();
  if (!dims_ok(Din, D)) TD_FAIL(TD_ERR_UNSUPPORTED, "td_aligner_bwd_dh2: Din=%d, D=%d must be multiples of 64 (D <= 4096)", Din, D);
  if (M <= 0 || M > 0x7fffffffll / D) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: M=%lld out of range", (long long)M);
  if (ws_bytes < td_aligner_bwd_workspace_bytes(M, Din, D)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: workspace too small");
  if (accumulate && sc) TD_FAIL(TD_ERR_UNSUPPORTED, "td_aligner_bwd_dh2_scatter: gradient accumulation needs local outputs");
  cudaStream_t st = (cudaStream_t)stream;
  BwdWorkspace w = carve_bwd(ws, M, D);
  if ((phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_W2_ONLY)) && (!dh2 || !h1 || !dW2))
    TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: null pointer (dW2)");
  NormPartials np;
  BwdExtras ex;
  ex.stats = stats; ex.accumulate = accumulate;
  if ((phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_SMALL2_ONLY)) || loss_out) {
    if (!norm_partials) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: norm_partials is null");
    if ((phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_SMALL2_ONLY)) && (!db2 || !dg)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: null pointer (dg / db2)");
    np = carve_norm_partials(const_cast<void*>(norm_partials), M, D);
    ex.np = &np;
    ex.loss_out = loss_out;
    ex.loss_div = float(M) * float(D);
  }
  if ((phases & TD_BWD_PHASE_GELU_W1) && (!x || !h0 || !W2 || !dW1 || !db1)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: null pointer (phase 2)");
  if ((phases & TD_BWD_PHASE_GELU_ONLY) && (!dh2 || !h0 || !W2 || !db1)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: null pointer (dh0 / db1)");
  if ((phases & TD_BWD_PHASE_W1_ONLY) && (!x || !dW1)) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2: null pointer (dW1)");
  return bwd_from_dh2(static_cast<const __nv_bfloat16*>(dh2), x, h0, h1, W2, M, Din, D, grad_scale, grad_scale_ptr, dW1, db1,
                      dW2, db2, dg, w, phases, st, sc, ex);
}
}  // namespace
extern "C" {

int32_t td_aligner_bwd_dh2(const void* dh2, const void* x, const void* h0, const void* h1, const void* W2,
                           const void* norm_partials, int64_t M, int32_t Din, int32_t D,
                           float grad_scale, const float* grad_scale_ptr, float* dW1, float* db1, float* dW2, float* db2,
                           float* dg, float* loss_out, float* stats, int32_t accumulate, void* ws, int64_t ws_bytes,
                           int32_t phases, td_stream_t stream) {
  return bwd_dh2_impl(dh2, x, h0, h1, W2, norm_partials, M, Din, D, grad_scale, grad_scale_ptr, dW1, db1, dW2, db2, dg, loss_out,
                      stats, accumulate, ws, ws_bytes, phases, stream, nullptr);
}

int32_t td_aligner_bwd_dh2_scatter(const void* dh2, const void* x, const void* h0, const void* h1, const void* W2,
                                   const void* norm_partials, int64_t M, int32_t Din, int32_t D, float grad_scale,
                                   const float* grad_scale_ptr, float* const* dW1_dst, float* db1, float* const* dW2_dst,
                                   float* db2, float* dg, float* loss_out, float* stats, int32_t world, int32_t rank,
                                   const td_peer_fold* fold, void* ws, int64_t ws_bytes, int32_t phases, td_stream_t stream) {
  if (world < 1 || world > kMaxPeers || D % world)
    TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: world=%d must be 1..%d and divide D=%d", world, kMaxPeers, D);
  if (rank >= world) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: rank=%d outside world=%d", rank, world);
  ScatterDst sc;
  sc.world = world;
  sc.rank = rank;
  const bool need1 = (phases & (TD_BWD_PHASE_GELU_W1 | TD_BWD_PHASE_W1_ONLY)) != 0;
  const bool need2 = (phases & (TD_BWD_PHASE_NORM_W2 | TD_BWD_PHASE_W2_ONLY)) != 0;
  for (int o = 0; o < world; ++o) {
    if ((need1 && (!dW1_dst || !dW1_dst[o])) || (need2 && (!dW2_dst || !dW2_dst[o])))
      TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: null destination for rank %d", o);
    if (need1) sc.dW1[o] = dW1_dst[o];
    if (need2) sc.dW2[o] = dW2_dst[o];
  }
  if (fold != nullptr) {
    if (fold->signal_flags != nullptr) {
      if (!(need1 || need2) || fold->signal_slot < 0) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: a folded signal needs a weight-gradient GEMM in this call");
      for (int o = 0; o < world; ++o) {
        if (!fold->signal_flags[o]) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: null flag array for rank %d", o);
        sc.signal[o] = static_cast<int*>(fold->signal_flags[o]) + fold->signal_slot;
      }
      sc.n_signal = world;
    }
    if (fold->small_dst != nullptr) {
      if (!fold->small_base || fold->small_numel <= 0) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: small_dst needs small_base / small_numel");
      for (int o = 0; o < world; ++o) {
        if (!fold->small_dst[o]) TD_FAIL(TD_ERR_ARG, "td_aligner_bwd_dh2_scatter: null small-vector slot for rank %d", o);
        sc.post[o] = static_cast<float*>(fold->small_dst[o]);
      }
      sc.n_post = world; sc.post_base = fold->small_base; sc.post_numel = fold->small_numel;
    }
  }
  // the impl's null checks look at dW1 / dW2: hand it the first destination
  return bwd_dh2_impl(dh2, x, h0, h1, W2, norm_partials, M, Din, D, grad_scale, grad_scale_ptr, need1 ? sc.dW1[0] : nullptr,
                      db1, need2 ? sc.dW2[0] : nullptr, db2, dg, loss_out, stats, 0, ws, ws_bytes, phases, stream, &sc);
}

// ------------------------------------------------------------------------------------------------ optimizer
namespace {
// torch computes the bias corrections in double (1 - beta ** step); so do we, on the host
inline void bias_corrections(float beta1, float beta2, int64_t step, float* c1, float* sqrt_c2) {
  *c1 = float(1.0 - std::pow((double)beta1, (double)step));
  *sqrt_c2 = float(std::sqrt(1.0 - std::pow((double)beta2, (double)step)));
}
}  // namespace

int32_t td_adamw_step(int32_t num_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                      float* const* exp_avg_sq, void* const* params_bf16, const int64_t* numel, const float* weight_decay,
                      float lr, float beta1, float beta2, float eps, int64_t step, float grad_scale, const void* step_ctl,
                      td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (num_tensors < 1 || num_tensors > 3) TD_FAIL(TD_ERR_ARG, "td_adamw_step: 1..3 tensors per call, got %d", num_tensors);
  if (step < 1 && !step_ctl) TD_FAIL(TD_ERR_ARG, "td_adamw_step: step counts from 1");
  AdamParams a;
  memset(&a, 0, sizeof(a));
  long long max_n = 0;
  bool wide = true;  // every tensor a multiple of 8 elements at 32-byte aligned addresses: 256-bit kernel
  for (int i = 0; i < num_tensors; ++i) {
    if (!params[i] || !grads[i] || !exp_avg[i] || !exp_avg_sq[i] || numel[i] < 0) TD_FAIL(TD_ERR_ARG, "td_adamw_step: null pointer");
    if (numel[i] % 4) TD_FAIL(TD_ERR_UNSUPPORTED, "td_adamw_step: tensor sizes must be multiples of 4 (got %lld)", (long long)numel[i]);
    const uintptr_t bits = reinterpret_cast<uintptr_t>(params[i]) | reinterpret_cast<uintptr_t>(grads[i]) |
                           reinterpret_cast<uintptr_t>(exp_avg[i]) | reinterpret_cast<uintptr_t>(exp_avg_sq[i]);
    if (bits & 15) TD_FAIL(TD_ERR_ARG, "td_adamw_step: buffers must be 16-byte aligned");
    const uintptr_t b16 = reinterpret_cast<uintptr_t>(params_bf16 ? params_bf16[i] : nullptr);
    wide = wide && !(bits & 31) && !(b16 & 15) && numel[i] % 8 == 0;
    a.seg[i] = AdamSegment{params[i], grads[i], exp_avg[i], exp_avg_sq[i],
                           static_cast<__nv_bfloat16*>(params_bf16 ? params_bf16[i] : nullptr), numel[i], weight_decay[i]};
    if (numel[i] > max_n) max_n = numel[i];
  }
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.grad_scale = grad_scale;
  a.ctl = static_cast<const StepCtl*>(step_ctl);
  bias_corrections(beta1, beta2, step < 1 ? 1 : step, &a.bias_c1, &a.sqrt_bias_c2);
  if (max_n == 0) return TD_OK;
  double total = 0;
  for (int i = 0; i < num_tensors; ++i) total += double(numel[i]);
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof("adamw_bf16", 30.0 * total, st);
  // 2 CTAs per SM: a wave of them fits beside a resident GEMM CTA (registers: 320 x 128 + 256 x 64), the second wave takes the
  // SM over as soon as the GEMM's CTAs retire
  prefer_max_shared(adamw256_kernel);
  // TD_ADAMW: developer A/B of the launch shape -- "wide2" (default) = 256-bit kernel, 2 CTAs per SM; "wide8" = 256-bit, 8 per SM;
  // "narrow8" = the 128-bit kernel, 8 per SM
  static const int mode = [] {
    const char* e = getenv("TD_ADAMW");
    return !e ? 0 : !strcmp(e, "wide8") ? 1 : !strcmp(e, "narrow8") ? 2 : 0;
  }();
  if (wide && mode != 2) adamw256_kernel<<<dim3(grid_for_rows(max_n / 8, 256, mode == 1 ? 8 : 2), num_tensors), 256, 0, st>>>(a);
  else adamw_kernel<<<dim3(grid_for_rows(max_n / 4, 256, 8), num_tensors), 256, 0, st>>>(a);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int64_t td_step_ctl_bytes(void) { return (int64_t)align_up(sizeof(StepCtl), 64); }

int32_t td_step_ctl_init(void* step_ctl, float init_scale, int64_t step, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!step_ctl || !(init_scale > 0.f) || step < 0) TD_FAIL(TD_ERR_ARG, "td_step_ctl_init: bad arguments");
  StepCtl h;
  memset(&h, 0, sizeof(h));
  h.grad_mult = 1.0f / init_scale; h.scale = init_scale; h.step = float(step);
  h.bias_c1 = 1.f; h.sqrt_bias_c2 = 1.f;
  // (pageable source: the copy is staged by the runtime before the call returns)
  TD_CUDA(cudaMemcpyAsync(step_ctl, &h, sizeof(h), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return TD_OK;
}

int32_t td_step_ctl_update(void* step_ctl, const float* stats, int32_t use_scaler, float growth_factor, float backoff_factor,
                           int32_t growth_interval, float beta1, float beta2, float max_grad_norm, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!step_ctl) TD_FAIL(TD_ERR_ARG, "td_step_ctl_update: null control block");
  step_ctl_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(static_cast<StepCtl*>(step_ctl), stats, use_scaler, growth_factor, backoff_factor,
                                                     growth_interval, beta1, beta2, max_grad_norm);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_grad_stats(const float* grad, int64_t numel, float* stats, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (numel < 0 || !stats || (numel > 0 && !grad)) TD_FAIL(TD_ERR_ARG, "td_grad_stats: bad arguments");
  if (reinterpret_cast<uintptr_t>(grad) & 15) TD_FAIL(TD_ERR_ARG, "td_grad_stats: buffer must be 16-byte aligned");
  if (numel == 0) return TD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof("grad_stats", 4.0 * double(numel), st);
  grad_stats_kernel<<<grid_for_rows(numel / 4 + 1, 256, 8), 256, 0, st>>>(grad, numel, stats);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

// ------------------------------------------------------------------------------------------------ peer-memory data parallel
int32_t td_peer_alloc(int64_t bytes, void** ptr, uint8_t* handle) {
  TD_DEVICE_OR_RETURN();
  static_assert(sizeof(cudaIpcMemHandle_t) == TD_IPC_HANDLE_BYTES, "IPC handle size");
  if (bytes <= 0 || !ptr || !handle) TD_FAIL(TD_ERR_ARG, "td_peer_alloc: bad arguments");
  void* p = nullptr;
  TD_CUDA(cudaMalloc(&p, (size_t)bytes));
  cudaError_t e = cudaMemset(p, 0, (size_t)bytes);  // flags start at step 0
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    TD_FAIL(-100 - int(e), "td_peer_alloc: %s", cudaGetErrorString(e));
  }
  memcpy(handle, &h, sizeof(h));
  *ptr = p;
  return TD_OK;
}

int32_t td_peer_free(void* ptr) {
  if (ptr) TD_CUDA(cudaFree(ptr));
  return TD_OK;
}

int32_t td_peer_open(const uint8_t* handle, void** ptr) {
  TD_DEVICE_OR_RETURN();
  if (!handle || !ptr) TD_FAIL(TD_ERR_ARG, "td_peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  TD_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return TD_OK;
}

int32_t td_peer_close(void* ptr) {
  if (ptr) TD_CUDA(cudaIpcCloseMemHandle(ptr));
  return TD_OK;
}

namespace {
int fill_peers(PeerPtrs& pp, void* const* arr, int n, const char* what) {
  memset(&pp, 0, sizeof(pp));
  if (n < 1 || n > kMaxPeers || !arr) TD_FAIL(TD_ERR_ARG, "%s: 1..%d destinations, got %d", what, kMaxPeers, n);
  for (int i = 0; i < n; ++i) {
    if (!arr[i]) TD_FAIL(TD_ERR_ARG, "%s: null pointer for rank %d", what, i);
    pp.p[i] = arr[i];
  }
  return TD_OK;
}
}  // namespace

int32_t td_peer_signal(void* const* flag_arrays, int32_t n, int32_t slot, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  PeerPtrs pp;
  int rc = fill_peers(pp, flag_arrays, n, "td_peer_signal");
  if (rc) return rc;
  if (slot < 0) TD_FAIL(TD_ERR_ARG, "td_peer_signal: negative slot");
  ProfScope prof("peer_signal", 0.0, (cudaStream_t)stream);
  peer_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(pp, n, slot);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

namespace {
// Stream memory operations (driver API, resolved at run time): the stream itself waits until a 32-bit word in device memory
// reaches a value -- no kernel, no SM, nothing that could keep a CTA pair of a persistent GEMM from becoming resident.
typedef CUresult (*PFN_streamWaitValue32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
inline PFN_streamWaitValue32 stream_wait_fn() {
  static PFN_streamWaitValue32 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* mode = getenv("TD_PEER_WAIT");
    if (mode && !strcmp(mode, "kernel")) return;  // developer override: the spinning wait kernel
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_streamWaitValue32>(p);
  });
  return fn;
}
}  // namespace

int32_t td_peer_wait(const int32_t* flags, int32_t n, int32_t value, float timeout_s, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!flags || n < 1 || n > 32) TD_FAIL(TD_ERR_ARG, "td_peer_wait: 1..32 flags");
  ProfScope prof("peer_wait", 0.0, (cudaStream_t)stream);  // (events around the wait: its span in the timeline is time spent blocked)
  if (PFN_streamWaitValue32 wait = stream_wait_fn()) {
    // flags only ever grow (counters): "*addr - value >= 0" is the condition CU_STREAM_WAIT_VALUE_GEQ tests
    for (int i = 0; i < n; ++i) {
      CUresult r = wait((CUstream)stream, (CUdeviceptr)(uintptr_t)(flags + i), (cuuint32_t)value, CU_STREAM_WAIT_VALUE_GEQ);
      if (r != CUDA_SUCCESS) TD_FAIL(TD_ERR_DRIVER, "cuStreamWaitValue32 failed with CUresult %d", int(r));
    }
    return TD_OK;
  }
  if (!(timeout_s > 0.f)) timeout_s = 600.f;
  peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, n, value, (unsigned long long)(double(timeout_s) * 1e9));
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_peer_post(const float* src, void* const* dst, int32_t n, int64_t numel, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  PeerPtrs pp;
  int rc = fill_peers(pp, dst, n, "td_peer_post");
  if (rc) return rc;
  if (!src || numel < 0 || numel % 4) TD_FAIL(TD_ERR_ARG, "td_peer_post: numel must be a non-negative multiple of 4");
  if (numel == 0) return TD_OK;
  ProfScope prof("peer_post", 4.0 * double(numel) * n, (cudaStream_t)stream);
  peer_post_kernel<<<grid_for_rows(numel / 4, 256, 2), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(src), pp, n, numel / 4);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_sum_slots(const float* slots, int64_t slot_stride, int32_t n_slots, float* out, int64_t numel, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!slots || !out || n_slots < 1 || numel < 0 || numel % 4 || slot_stride % 4 || slot_stride < numel)
    TD_FAIL(TD_ERR_ARG, "td_sum_slots: bad arguments (numel and slot_stride must be multiples of 4, slot_stride >= numel)");
  if (numel == 0) return TD_OK;
  sum_slots_kernel<<<grid_for_rows(numel / 4, 256, 4), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(slots), slot_stride / 4, n_slots, reinterpret_cast<float4*>(out), numel / 4);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_adamw_slots_step(float* param, const float* grad_slots, int64_t slot_stride, int32_t n_slots, float* exp_avg,
                            float* exp_avg_sq, void* const* params_bf16, int32_t n_dst, int64_t numel, float weight_decay,
                            float lr, float beta1, float beta2, float eps, int64_t step, float grad_scale,
                            const void* step_ctl, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (!param || !grad_slots || !exp_avg || !exp_avg_sq || numel < 0) TD_FAIL(TD_ERR_ARG, "td_adamw_slots_step: null pointer");
  if (numel % 4 || slot_stride % 4 || slot_stride < numel || n_slots < 1)
    TD_FAIL(TD_ERR_ARG, "td_adamw_slots_step: numel / slot_stride must be multiples of 4, slot_stride >= numel, n_slots >= 1");
  if (step < 1 && !step_ctl) TD_FAIL(TD_ERR_ARG, "td_adamw_slots_step: step counts from 1");
  AdamSlotsParams a;
  memset(&a, 0, sizeof(a));
  int rc = fill_peers(a.p_bf16, params_bf16, n_dst, "td_adamw_slots_step");
  if (rc) return rc;
  a.p = param; a.m = exp_avg; a.v = exp_avg_sq; a.slots = grad_slots; a.slot_stride = slot_stride; a.n_slots = n_slots;
  a.n_dst = n_dst; a.n = numel; a.weight_decay = weight_decay;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.grad_scale = grad_scale;
  a.ctl = static_cast<const StepCtl*>(step_ctl);
  bias_corrections(beta1, beta2, step < 1 ? 1 : step, &a.bias_c1, &a.sqrt_bias_c2);
  if (numel == 0) return TD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof("adamw_slots", (28.0 + 4.0 * n_slots + 2.0 * n_dst) * double(numel), st);
  prefer_max_shared(adamw_slots_kernel);
  adamw_slots_kernel<<<grid_for_rows(numel / 4, 256, 2), 256, 0, st>>>(a);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

}  // extern "C"
namespace {
struct SegmentRecorder {  // (a functor rather than a lambda: for_each_segment is __host__ __device__)
  int32_t* out; int max; int* n; int unit;
  __host__ __device__ void operator()(const Segment& s, int range) const {
    if (*n < max) {
      int32_t* o = out + 8 * *n;
      o[0] = unit; o[1] = s.tile; o[2] = s.kb0; o[3] = s.kb1; o[4] = s.kind; o[5] = s.contrib0; o[6] = s.contrib_n; o[7] = range;
    }
    ++*n;
  }
};
}  // namespace
extern "C" {

int32_t td_gemm_schedule(int64_t M, int32_t N, int64_t K, int32_t workers, int32_t stream_k, int32_t* out, int32_t max_segments) {
  // host arithmetic only: plan_schedule() + for_each_segment(), the code the launch and the kernel run
  if (M <= 0 || N <= 0 || K <= 0 || workers < 1 || M > 0x7fffffffll || K > 0x7fffffffll || (max_segments > 0 && !out)) return -1;
  GemmParams p = gemm_params(M, N, K);
  set_tile_grid(p, 2);  // a CTA-pair GEMM, as every composite entry launches
  plan_schedule(p, workers, stream_k != 0);
  int n = 0;
  const int units = num_units(p);
  for (int u = 0; u < units; ++u) for_each_segment(p, u, SegmentRecorder{out, max_segments, &n, u});
  return n;
}

int32_t td_scatter_tile_owner(int32_t tile, int32_t M, int32_t N, int32_t world, int32_t rank, int32_t* m_blk_out, int32_t* n_blk_out) {
  // host arithmetic only (no device needed): the same tile_coords() the kernel runs, with the raster launch_dw_gemm sets up
  if (M <= 0 || N <= 0 || world < 1 || world > kMaxPeers || M % world || (M / world) % 32 || rank >= world) return -1;
  GemmParams p = gemm_params(M, N, 0);
  set_tile_grid(p, 2);  // launch_dw_gemm runs CTA pairs
  if (tile < 0 || tile >= p.num_m_blocks * p.num_n_blocks) return -1;
  set_scatter_raster(p, world, rank);
  int m_blk = 0, n_blk = 0;
  tile_coords(p, tile, m_blk, n_blk);
  if (m_blk_out) *m_blk_out = m_blk;
  if (n_blk_out) *n_blk_out = n_blk;
  return (m_blk * 2 * kBlockM) / p.scatter_rows;
}

int32_t td_gemm_tn_scatter(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int32_t N, int64_t K, float alpha,
                           float* const* dst, int32_t world, int32_t rank, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (rank >= world) TD_FAIL(TD_ERR_ARG, "td_gemm_tn_scatter: rank=%d outside world=%d", rank, world);
  if (world < 1 || world > kMaxPeers || M % world) TD_FAIL(TD_ERR_ARG, "td_gemm_tn_scatter: world=%d must be 1..%d and divide M", world, kMaxPeers);
  if (M <= 0 || M > 0x7fffffffll || K <= 0 || K > 0x7fffffffll) TD_FAIL(TD_ERR_ARG, "td_gemm_tn_scatter: size out of range");
  GemmParams p = gemm_params(M, N, K);
  p.alpha = alpha;
  for (int o = 0; o < world; ++o) {
    if (!dst || !dst[o]) TD_FAIL(TD_ERR_ARG, "td_gemm_tn_scatter: null destination for rank %d", o);
  }
  return launch_dw_gemm({A, lda, true}, {B, ldb, true}, p, dst, world, rank, sk_ws_or_null(ws, ws_bytes), (cudaStream_t)stream, "gemm_tn_scatter");
}

// ------------------------------------------------------------------------------------------------ losses
int64_t td_loss_workspace_bytes(int64_t rows) {
  const size_t parts = (size_t)device_sm_count() * 8 + 8;
  return (int64_t)(align_up(sizeof(float) * 8, 256) + align_up(sizeof(float) * parts, 256) +
                   align_up(sizeof(float) * (size_t)(rows > 0 ? rows : 1), 256));
}

int32_t td_masked_mse_fwd_bwd(const void* y, int32_t y_dtype, const void* t, int32_t t_dtype, const int64_t* row_mask,
                              int64_t M, int32_t D, float grad_scale, float* loss, void* dy, void* ws, int64_t ws_bytes,
                              td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (M < 0 || D <= 0 || D % 8) TD_FAIL(TD_ERR_ARG, "td_masked_mse_fwd_bwd: D=%d must be a positive multiple of 8", D);
  if (!loss) TD_FAIL(TD_ERR_ARG, "td_masked_mse_fwd_bwd: loss pointer is null");
  if (ws_bytes < td_loss_workspace_bytes(M)) TD_FAIL(TD_ERR_ARG, "td_masked_mse_fwd_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  Carver c(ws);
  float* meta = c.take<float>(8);
  float* part = c.take<float>((size_t)device_sm_count() * 8 + 8);
  count_valid_kernel<<<1, 1024, 0, st>>>(reinterpret_cast<const long long*>(row_mask), M, 0, meta);
  int grid = 1;
  if (M > 0) {
    grid = grid_for_rows(M, 8, 8);
    const long long* mk = reinterpret_cast<const long long*>(row_mask);
    const int sel = (y_dtype == TD_DTYPE_BF16 ? 2 : 0) | (t_dtype == TD_DTYPE_BF16 ? 1 : 0);
    ProfScope prof("masked_mse", double(M) * D * ((y_dtype == TD_DTYPE_BF16 ? 2.0 : 4.0) * (dy ? 2.0 : 1.0) + (t_dtype == TD_DTYPE_BF16 ? 2.0 : 4.0)), st);
    switch (sel) {
      case 0: masked_mse_kernel<false, false><<<grid, 256, 0, st>>>(y, t, mk, int(M), D, meta, grad_scale, dy, part); break;
      case 1: masked_mse_kernel<false, true><<<grid, 256, 0, st>>>(y, t, mk, int(M), D, meta, grad_scale, dy, part); break;
      case 2: masked_mse_kernel<true, false><<<grid, 256, 0, st>>>(y, t, mk, int(M), D, meta, grad_scale, dy, part); break;
      default: masked_mse_kernel<true, true><<<grid, 256, 0, st>>>(y, t, mk, int(M), D, meta, grad_scale, dy, part); break;
    }
  } else {
    TD_CUDA(cudaMemsetAsync(part, 0, sizeof(float), st));
  }
  loss_finish_kernel<<<1, 256, 0, st>>>(part, grid, meta, float(D), loss);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

int32_t td_masked_ce_fwd_bwd(const void* logits, int32_t dtype, const int64_t* labels, int64_t R, int32_t V,
                             float grad_scale, float* loss, void* dlogits, void* ws, int64_t ws_bytes,
                             td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (R < 0 || V <= 0 || V % 8) TD_FAIL(TD_ERR_ARG, "td_masked_ce_fwd_bwd: V=%d must be a positive multiple of 8", V);
  if ((size_t)V * sizeof(float) > 200 * 1024) TD_FAIL(TD_ERR_UNSUPPORTED, "td_masked_ce_fwd_bwd: V=%d does not fit the smem row stage", V);
  if (!loss || (R > 0 && (!logits || !labels))) TD_FAIL(TD_ERR_ARG, "td_masked_ce_fwd_bwd: null pointer");
  if (ws_bytes < td_loss_workspace_bytes(R)) TD_FAIL(TD_ERR_ARG, "td_masked_ce_fwd_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  Carver c(ws);
  float* meta = c.take<float>(8);
  (void)c.take<float>((size_t)device_sm_count() * 8 + 8);
  float* row_loss = c.take<float>((size_t)(R > 0 ? R : 1));
  count_valid_kernel<<<1, 1024, 0, st>>>(reinterpret_cast<const long long*>(labels), R, 1, meta);
  if (R > 0) {
    const size_t smem = (size_t)V * (dtype == TD_DTYPE_BF16 ? 2 : 4);  // the row is staged in its input dtype
    ProfScope prof("masked_ce", double(R) * V * (dtype == TD_DTYPE_BF16 ? 2.0 : 4.0) * (dlogits ? 2.0 : 1.0), st);
    static std::atomic<bool> attr_done_dev[2][kMaxDevices];  // (function attributes are per device)
    const int dev = current_device();
    if (dev < 0 || dev >= kMaxDevices) TD_FAIL(TD_ERR_DRIVER, "no current CUDA device");
    std::atomic<bool>* attr_done[2] = {&attr_done_dev[0][dev], &attr_done_dev[1][dev]};
    if (dtype == TD_DTYPE_BF16) {
      if (!attr_done[1]->load()) { TD_CUDA(cudaFuncSetAttribute(masked_ce_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); attr_done[1]->store(true); }
      masked_ce_kernel<true><<<int(R), kCeThreads, smem, st>>>(logits, reinterpret_cast<const long long*>(labels), V, meta, grad_scale, dlogits, row_loss);
    } else {
      if (!attr_done[0]->load()) { TD_CUDA(cudaFuncSetAttribute(masked_ce_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); attr_done[0]->store(true); }
      masked_ce_kernel<false><<<int(R), kCeThreads, smem, st>>>(logits, reinterpret_cast<const long long*>(labels), V, meta, grad_scale, dlogits, row_loss);
    }
    TD_CUDA(cudaGetLastError());
  } else {
    TD_CUDA(cudaMemsetAsync(row_loss, 0, sizeof(float), st));
  }
  loss_finish_kernel<<<1, 256, 0, st>>>(row_loss, int(R), meta, 1.0f, loss);
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

// ------------------------------------------------------------------------------------------------ lm_head + CE (8 f-1)
int64_t td_lm_head_ce_workspace_bytes(int64_t R) { return td_loss_workspace_bytes(R) + 256 + td_gemm_workspace_bytes(); }

int32_t td_lm_head_ce_fwd_bwd(const void* seq, int64_t R, int32_t K, const void* W_lm, int32_t V, const int64_t* labels,
                              float grad_scale, float* loss, void* logits, void* dlogits, void* dseq, void* ws, int64_t ws_bytes,
                              td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  if (R < 0 || K <= 0 || V <= 0 || K % 64 || V % 32) TD_FAIL(TD_ERR_UNSUPPORTED, "td_lm_head_ce_fwd_bwd: need K %% 64 == 0 and V %% 32 == 0 (K=%d V=%d)", K, V);
  if (!loss || (R > 0 && (!seq || !W_lm || !labels || !logits))) TD_FAIL(TD_ERR_ARG, "td_lm_head_ce_fwd_bwd: null pointer");
  if (dseq && !dlogits) TD_FAIL(TD_ERR_ARG, "td_lm_head_ce_fwd_bwd: dseq needs a dlogits buffer (it may alias logits)");
  if (!ws || ws_bytes < td_lm_head_ce_workspace_bytes(R)) TD_FAIL(TD_ERR_ARG, "td_lm_head_ce_fwd_bwd: workspace too small");
  const int64_t loss_bytes = (td_loss_workspace_bytes(R) + 255) / 256 * 256;
  char* sk = static_cast<char*>(ws) + loss_bytes;
  const int64_t sk_bytes = ws_bytes - loss_bytes;
  int rc = td_linear_bf16(seq, R, K, W_lm, V, nullptr, logits, sk, sk_bytes, stream);
  if (rc) return rc;
  rc = td_masked_ce_fwd_bwd(logits, TD_DTYPE_BF16, labels, R, V, grad_scale, loss, dlogits, ws, loss_bytes, stream);
  if (rc) return rc;
  if (dseq) rc = td_linear_bf16_dx(dlogits, R, V, W_lm, K, dseq, sk, sk_bytes, stream);
  return rc;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ T5 attention (8 f-1)
namespace {
struct AttnCall {
  int B, H, max_len_q, max_len_k;
  bool causal;
  AttnParams p;
};

// Host checks shared by the forward and the backward; fills the kernel parameters that both use.
int attn_check(const char* fn, const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const int32_t* cu_q,
               const int32_t* cu_k, int32_t B, int32_t H, int32_t inner, int32_t max_len_q, int32_t max_len_k, int64_t Mq,
               int32_t self_attention, const float* bias, int32_t n_dist, AttnCall& c) {
  if (B < 0 || B > 65535 || H <= 0 || H > 65535 || max_len_q < 0 || max_len_k < 0 || Mq < 0)
    TD_FAIL(TD_ERR_ARG, "%s: bad sizes (B=%d H=%d max_len_q=%d max_len_k=%d Mq=%lld)", fn, B, H, max_len_q, max_len_k, (long long)Mq);
  if (inner != kAttnDk * H) TD_FAIL(TD_ERR_UNSUPPORTED, "%s: inner=%d must be 64 * H = %d (d_kv = 64 only)", fn, inner, kAttnDk * H);
  // (self-attention reads cu_q for its keys too)
  int rc = check_pointers(fn, {{"q", q}, {"k", k}, {"v", v}, {"cu_q", cu_q, kNonNull}, {"cu_k", self_attention ? cu_q : cu_k, kNonNull}});
  if (rc) return rc;
  if (ldq % 8 || ldk % 8 || ldv % 8 || ldq < inner || ldk < inner || ldv < inner)
    TD_FAIL(TD_ERR_ARG, "%s: row pitches must be multiples of 8 and >= inner (ldq=%lld ldk=%lld ldv=%lld)", fn, (long long)ldq,
            (long long)ldk, (long long)ldv);
  if (self_attention) {
    if (!bias) TD_FAIL(TD_ERR_ARG, "%s: self-attention needs the relative position bias table", fn);
    if (cu_k && cu_k != cu_q) TD_FAIL(TD_ERR_ARG, "%s: self-attention attends to its own rows: cu_k must be NULL or cu_q", fn);
    if (n_dist < 1 || n_dist > kAttnMaxDist) TD_FAIL(TD_ERR_ARG, "%s: n_dist=%d must be in [1, %d]", fn, n_dist, kAttnMaxDist);
  } else if (bias) {
    TD_FAIL(TD_ERR_ARG, "%s: cross-attention takes no position bias", fn);
  }
  c.B = B; c.H = H; c.max_len_q = max_len_q; c.max_len_k = max_len_k; c.causal = self_attention != 0;
  memset(&c.p, 0, sizeof(c.p));
  c.p.q = static_cast<const __nv_bfloat16*>(q); c.p.k = static_cast<const __nv_bfloat16*>(k); c.p.v = static_cast<const __nv_bfloat16*>(v);
  c.p.ldq = ldq; c.p.ldk = ldk; c.p.ldv = ldv;
  c.p.cu_q = cu_q; c.p.cu_k = self_attention ? cu_q : cu_k;
  c.p.bias = self_attention ? bias : nullptr; c.p.n_dist = self_attention ? n_dist : 0;
  c.p.H = H; c.p.Mq = Mq;
  return TD_OK;
}

// Visible (query, key) pairs summed over the samples, for the profiler's FLOP count; 0 unless profiling is on (then it reads
// cu_* back, which synchronises the stream).
double attn_visible_pairs(const AttnCall& c, cudaStream_t st) {
  if (!Profiler::get().on.load(std::memory_order_relaxed) || c.B == 0) return 0.0;
  std::vector<int> hq(c.B + 1), hk(c.B + 1);
  if (cudaMemcpyAsync(hq.data(), c.p.cu_q, sizeof(int) * (c.B + 1), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaMemcpyAsync(hk.data(), c.p.cu_k, sizeof(int) * (c.B + 1), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess) {
    cudaGetLastError();
    return 0.0;
  }
  double pairs = 0.0;
  for (int b = 0; b < c.B; ++b) {
    const double T = hq[b + 1] - hq[b], L = hk[b + 1] - hk[b];
    pairs += c.causal ? T * (T + 1) / 2 : T * L;
  }
  return pairs;
}

template <class K>
int attn_launch(K kernel, dim3 grid, int threads, int smem, cudaStream_t st, const AttnParams& p, const char* tag, double work) {
  if (grid.x == 0 || grid.y == 0 || grid.z == 0) return TD_OK;
  TD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  {
    ProfScope prof(tag, work, st);
    kernel<<<grid, threads, smem, st>>>(p);
  }
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}

inline unsigned attn_tiles(int max_len) { return unsigned((max_len + kAttnTile - 1) / kAttnTile); }
}  // namespace

extern "C" int64_t td_t5_attention_workspace_bytes(int64_t Mq, int32_t H) {
  const size_t rows = (size_t)(Mq > 0 ? Mq : 1), heads = (size_t)(H > 0 ? H : 1);
  return (int64_t)align_up(sizeof(float) * rows * heads, 256);  // Delta [H, Mq]
}

namespace {
// Every check of the forward (attn_check and the output), run before anything is enqueued; attn_fwd_run then only launches.
int attn_fwd_check(const char* fn, const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const int32_t* cu_q,
                   const int32_t* cu_k, int32_t B, int32_t H, int32_t inner, int32_t max_len_q, int32_t max_len_k, int64_t Mq,
                   int32_t self_attention, const float* bias, int32_t n_dist, void* o, int64_t ldo, float* lse, AttnCall& c) {
  int rc = attn_check(fn, q, ldq, k, ldk, v, ldv, cu_q, cu_k, B, H, inner, max_len_q, max_len_k, Mq, self_attention, bias, n_dist, c);
  if (rc) return rc;
  rc = check_pointers(fn, {{"o", o}});
  if (rc) return rc;
  if (ldo % 8 || ldo < inner) TD_FAIL(TD_ERR_ARG, "%s: o's row pitch must be a multiple of 8 and >= inner (ldo=%lld)", fn, (long long)ldo);
  c.p.out = static_cast<__nv_bfloat16*>(o); c.p.ld_out = ldo; c.p.lse = lse;
  return TD_OK;
}

int attn_fwd_run(const AttnCall& c, cudaStream_t st) {
  const double flops = 4.0 * kAttnDk * c.H * attn_visible_pairs(c, st);
  const dim3 grid(attn_tiles(c.max_len_q), c.H, c.B);
  const int smem = attn_smem_bytes(AttnFwdSmem::kBias, c.p.n_dist);
  return attn_launch(c.causal ? t5_attn_fwd_kernel<true> : t5_attn_fwd_kernel<false>, grid, kAttnThreads, smem, st, c.p, "attn_fwd", flops);
}

// Every check of the backward; attn_bwd_run then launches the row sums of dO * O, dK / dV and dQ.
int attn_bwd_check(const char* fn, const void* dout, int64_t lddo, const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                   int64_t ldv, const int32_t* cu_q, const int32_t* cu_k, int32_t B, int32_t H, int32_t inner, int32_t max_len_q,
                   int32_t max_len_k, int64_t Mq, int32_t self_attention, const float* bias, int32_t n_dist, const void* o,
                   int64_t ldo, const float* lse, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                   void* ws, int64_t ws_bytes, AttnCall& c) {
  int rc = attn_check(fn, q, ldq, k, ldk, v, ldv, cu_q, cu_k, B, H, inner, max_len_q, max_len_k, Mq, self_attention, bias, n_dist, c);
  if (rc) return rc;
  rc = check_pointers(fn, {{"dout", dout}, {"o", o}, {"lse", lse, kNonNull}, {"dq", dq}, {"dk", dk}, {"dv", dv}});
  if (rc) return rc;
  if (lddo % 8 || ldo % 8 || lddq % 8 || lddk % 8 || lddv % 8 || lddo < inner || ldo < inner || lddq < inner || lddk < inner || lddv < inner)
    TD_FAIL(TD_ERR_ARG, "%s: row pitches must be multiples of 8 and >= inner", fn);
  if (!ws || ws_bytes < td_t5_attention_workspace_bytes(Mq, H)) TD_FAIL(TD_ERR_ARG, "%s: workspace too small", fn);
  c.p.dout = static_cast<const __nv_bfloat16*>(dout); c.p.lddo = lddo;
  c.p.o = static_cast<const __nv_bfloat16*>(o); c.p.ldo = ldo;
  c.p.lse = const_cast<float*>(lse);
  c.p.delta = static_cast<float*>(ws);
  c.p.dq = static_cast<__nv_bfloat16*>(dq); c.p.lddq = lddq;
  c.p.dk = static_cast<__nv_bfloat16*>(dk); c.p.lddk = lddk;
  c.p.dv = static_cast<__nv_bfloat16*>(dv); c.p.lddv = lddv;
  return TD_OK;
}

int attn_bwd_run(const AttnCall& c, cudaStream_t st) {
  if (c.B == 0) return TD_OK;
  const int H = c.H;
  const long long Mq = c.p.Mq;
  const double pairs = attn_visible_pairs(c, st);
  const long long delta_threads = Mq * H * 8;
  int rc = attn_launch(t5_attn_delta_kernel, dim3(unsigned((delta_threads + 255) / 256)), 256, 0, st, c.p, "attn_bwd_delta",
                       double(Mq) * H * (4.0 * kAttnDk + 4.0));
  if (rc) return rc;
  const dim3 grid_k(attn_tiles(c.max_len_k), H, c.B), grid_q(attn_tiles(c.max_len_q), H, c.B);
  const int smem_kv = attn_smem_bytes(AttnDkdvSmem::kBias, c.p.n_dist), smem_q = attn_smem_bytes(AttnDqSmem::kBias, c.p.n_dist);
  const double f = 2.0 * kAttnDk * H * pairs;
  rc = attn_launch(c.causal ? t5_attn_dkdv_kernel<true> : t5_attn_dkdv_kernel<false>, c.causal ? grid_q : grid_k, kAttnThreads, smem_kv, st,
                   c.p, "attn_bwd_dkdv", 4 * f);
  if (rc) return rc;
  return attn_launch(c.causal ? t5_attn_dq_kernel<true> : t5_attn_dq_kernel<false>, grid_q, kAttnThreads, smem_q, st, c.p, "attn_bwd_dq", 3 * f);
}
}  // namespace

extern "C" {

int32_t td_t5_attention_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const int32_t* cu_q,
                            const int32_t* cu_k, int32_t B, int32_t H, int32_t inner, int32_t max_len_q, int32_t max_len_k, int64_t Mq,
                            int32_t self_attention, const float* bias, int32_t n_dist, void* o, int64_t ldo, float* lse,
                            td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  AttnCall c;
  int rc = attn_fwd_check("td_t5_attention_fwd", q, ldq, k, ldk, v, ldv, cu_q, cu_k, B, H, inner, max_len_q, max_len_k, Mq,
                          self_attention, bias, n_dist, o, ldo, lse, c);
  return rc ? rc : attn_fwd_run(c, (cudaStream_t)stream);
}

int32_t td_t5_attention_bwd(const void* dout, int64_t lddo, const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                            int64_t ldv, const int32_t* cu_q, const int32_t* cu_k, int32_t B, int32_t H, int32_t inner, int32_t max_len_q,
                            int32_t max_len_k, int64_t Mq, int32_t self_attention, const float* bias, int32_t n_dist, const void* o,
                            int64_t ldo, const float* lse, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                            void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  AttnCall c;
  int rc = attn_bwd_check("td_t5_attention_bwd", dout, lddo, q, ldq, k, ldk, v, ldv, cu_q, cu_k, B, H, inner, max_len_q, max_len_k, Mq,
                          self_attention, bias, n_dist, o, ldo, lse, dq, lddq, dk, lddk, dv, lddv, ws, ws_bytes, c);
  return rc ? rc : attn_bwd_run(c, (cudaStream_t)stream);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ T5 gated-GELU FFN (8 f-1)
namespace {
// Workspace of td_t5_ffn_fwd / _bwd: a [M, d] bf16 row buffer (xn forward, dxn backward), a [M, 2 d_ff] bf16 buffer (gated forward,
// d_ab backward, each when the caller passes none) and the stream-K tail of the GEMMs, which run one after another on the stream.
struct FfnWorkspace {
  __nv_bfloat16* rows;
  __nv_bfloat16* pairs;
  void* sk;
  size_t bytes;
};
FfnWorkspace carve_ffn(void* ws, int64_t M, int32_t d, int32_t d_ff) {
  const size_t m = (size_t)(M > 0 ? M : 1);
  Carver c(ws);
  FfnWorkspace w;
  w.rows = c.take<__nv_bfloat16>(m * (size_t)(d > 0 ? d : 1));
  w.pairs = c.take<__nv_bfloat16>(m * 2 * (size_t)(d_ff > 0 ? d_ff : 1));
  w.sk = c.take<uint8_t>(gemm_sk_workspace_bytes());
  w.bytes = c.off;
  return w;
}

int ffn_check_sizes(const char* fn, int64_t M, int32_t d, int32_t d_ff) {
  if (M < 0 || d <= 0 || d_ff <= 0) TD_FAIL(TD_ERR_ARG, "%s: bad sizes (M=%lld d=%d d_ff=%d)", fn, (long long)M, d, d_ff);
  if (d % 64 || d > 8 * kNormBwdThreads || d_ff % 32)
    TD_FAIL(TD_ERR_UNSUPPORTED, "%s: need d %% 64 == 0, d <= %d and d_ff %% 32 == 0 (d=%d d_ff=%d)", fn, 8 * kNormBwdThreads, d, d_ff);
  if (M > 0x7fffffffll / (2ll * d_ff)) TD_FAIL(TD_ERR_ARG, "%s: M=%lld out of range", fn, (long long)M);
  return TD_OK;
}
int ffn_check_workspace(const char* fn, int64_t M, int32_t d, int32_t d_ff, void* ws, int64_t ws_bytes) {
  if (!ws || ws_bytes < (int64_t)carve_ffn(nullptr, M, d, d_ff).bytes) TD_FAIL(TD_ERR_ARG, "%s: workspace too small", fn);
  return check_pointers(fn, {{"the workspace", ws, kOptionalAligned}});
}

// dx = bf16(dy + norm_bwd(dxn)): the backward of a T5 pre-norm sublayer's RMSNorm with the residual gradient folded in, one launch.
// Shared by the FFN and both attention sublayers; ln_w is frozen, so no weight-gradient partials are formed.
int residual_norm_bwd_launch(const __nv_bfloat16* dxn, const void* x, const float* rstd, const float* ln_w, int64_t M, int32_t d,
                             const void* dy, void* dx, const char* tag, cudaStream_t st) {
  int rpc;
  const int grid = norm_grid(M, 2, &rpc);
  {
    ProfScope prof(tag, double(M) * d * 8.0, st);
    rmsnorm_bwd_kernel<true, true><<<grid, kNormBwdThreads, 0, st>>>(dxn, static_cast<const __nv_bfloat16*>(x), rstd, ln_w, int(M), d,
                                                                     rpc, static_cast<__nv_bfloat16*>(dx), nullptr, nullptr,
                                                                     static_cast<const __nv_bfloat16*>(dy));
  }
  TD_CUDA(cudaGetLastError());
  return TD_OK;
}
}  // namespace

extern "C" {

int64_t td_t5_ffn_workspace_bytes(int64_t M, int32_t d, int32_t d_ff) { return (int64_t)carve_ffn(nullptr, M, d, d_ff).bytes; }

int32_t td_t5_ffn_fwd(const void* x, int64_t M, int32_t d, int32_t d_ff, const float* ln_w, float eps, const void* wi, const void* wo,
                      void* out, float* rstd, void* ab, void* gated, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  int rc = ffn_check_sizes("td_t5_ffn_fwd", M, d, d_ff);
  if (rc) return rc;
  if (M == 0) return TD_OK;
  rc = ffn_check_workspace("td_t5_ffn_fwd", M, d, d_ff, ws, ws_bytes);
  if (rc) return rc;
  rc = check_pointers("td_t5_ffn_fwd", {{"x", x}, {"ln_w", ln_w}, {"wi", wi}, {"wo", wo}, {"out", out}, {"rstd", rstd, kNonNull},
                                        {"ab", ab, kOptionalAligned}, {"gated", gated, kOptionalAligned}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const FfnWorkspace w = carve_ffn(ws, M, d, d_ff);
  __nv_bfloat16* xn = w.rows;
  void* g = gated ? gated : w.pairs;
  rc = rmsnorm_fwd_launch(x, nullptr, 0, ln_w, eps, M, d, xn, TD_DTYPE_BF16, rstd, "ffn_norm", st);
  if (rc) return rc;
  GemmParams p = gemm_params(M, 2 * d_ff, d);
  p.out0 = ab; p.out1 = g;
  rc = launch_gemm<2, false, false, EPI_GATED>({xn, d, false}, {wi, d, false}, p, w.sk, st, "gemm_ffn_gate");
  if (rc) return rc;
  return gemm_residual(g, M, d_ff, wo, d, x, out, w.sk, st, "gemm_ffn_out");
}

int32_t td_t5_ffn_bwd(const void* dy, const void* x, const float* rstd, const float* ln_w, const void* ab, const void* wi, const void* wo,
                      int64_t M, int32_t d, int32_t d_ff, void* dx, void* d_ab, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  int rc = ffn_check_sizes("td_t5_ffn_bwd", M, d, d_ff);
  if (rc) return rc;
  if (M == 0) return TD_OK;
  rc = ffn_check_workspace("td_t5_ffn_bwd", M, d, d_ff, ws, ws_bytes);
  if (rc) return rc;
  rc = check_pointers("td_t5_ffn_bwd", {{"dy", dy}, {"x", x}, {"rstd", rstd, kNonNull}, {"ln_w", ln_w, kNonNull}, {"ab", ab}, {"wi", wi},
                                        {"wo", wo}, {"dx", dx}, {"d_ab", d_ab, kOptionalAligned}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const FfnWorkspace w = carve_ffn(ws, M, d, d_ff);
  void* dab = d_ab ? d_ab : w.pairs;
  __nv_bfloat16* dxn = w.rows;
  GemmParams p = gemm_params(M, d_ff, d);  // t = dy . wo, wo [d, d_ff] read MN-major in place
  p.out0 = dab; p.aux0 = ab; p.ld_out = 2 * d_ff;
  rc = launch_gemm<2, false, true, EPI_DGATED>({dy, d, false}, {wo, d_ff, true}, p, w.sk, st, "gemm_ffn_dgate");
  if (rc) return rc;
  // dxn = d_ab . wi, over the interleaved pair columns of both
  rc = gemm_linear_dx(dab, M, 2 * d_ff, wi, d, dxn, false, w.sk, st, "gemm_ffn_dx");
  if (rc) return rc;
  return residual_norm_bwd_launch(dxn, x, rstd, ln_w, M, d, dy, dx, "ffn_norm_bwd", st);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ T5 attention sublayers (8 f-1)
namespace {
// Workspace of td_t5_{self,cross}_attention_layer_fwd / _bwd; every buffer serves the forward and then the backward:
//   rows  [M, d] bf16             xn / dxn
//   proj  [M, 3 inner] bf16       qkv / dqkv (self; when the caller passes none), or [Mk, 2 inner] kv / dkv (cross; kv when none given)
//   q     [M, inner] bf16         cross only: q (when none given) / dq
//   heads [M, inner] bf16         o (when none given) / d_o
//   rstd  [M] fp32                when the caller passes none
//   delta [H, M] fp32             the attention backward's row sums (td_t5_attention_workspace_bytes)
// and the stream-K tail of the GEMMs, which run one after another on the stream.
struct AttnLayerWorkspace {
  __nv_bfloat16 *rows, *proj, *q, *heads;
  float *rstd, *delta;
  int64_t delta_bytes;
  void* sk;
  size_t bytes;
};
AttnLayerWorkspace carve_attn_layer(void* ws, int64_t M, int64_t Mk, int32_t d, int32_t H, bool self_attention) {
  const size_t m = (size_t)(M > 0 ? M : 1), mk = (size_t)(Mk > 0 ? Mk : 1), dd = (size_t)(d > 0 ? d : 1);
  const size_t inner = (size_t)kAttnDk * (H > 0 ? H : 1);
  Carver c(ws);
  AttnLayerWorkspace w;
  w.rows = c.take<__nv_bfloat16>(m * dd);
  w.proj = c.take<__nv_bfloat16>(self_attention ? m * 3 * inner : mk * 2 * inner);
  w.q = self_attention ? nullptr : c.take<__nv_bfloat16>(m * inner);
  w.heads = c.take<__nv_bfloat16>(m * inner);
  w.rstd = c.take<float>(m);
  w.delta_bytes = td_t5_attention_workspace_bytes(M, H);
  w.delta = c.take<float>((size_t)w.delta_bytes / sizeof(float));
  w.sk = c.take<uint8_t>(gemm_sk_workspace_bytes());
  w.bytes = c.off;
  return w;
}

int attn_layer_check(const char* fn, int64_t M, int64_t Mk, int32_t d, int32_t H, bool self_attention, void* ws, int64_t ws_bytes) {
  if (M < 0 || Mk < 0 || d <= 0 || H <= 0 || H > 65535)
    TD_FAIL(TD_ERR_ARG, "%s: bad sizes (M=%lld Mk=%lld d=%d H=%d)", fn, (long long)M, (long long)Mk, d, H);
  if (d % 64 || d > 8 * kNormBwdThreads) TD_FAIL(TD_ERR_UNSUPPORTED, "%s: need d %% 64 == 0 and d <= %d (d=%d)", fn, 8 * kNormBwdThreads, d);
  const long long widest = 3ll * kAttnDk * H > d ? 3ll * kAttnDk * H : (long long)d;
  if (M > 0x7fffffffll / widest || Mk > 0x7fffffffll / widest)
    TD_FAIL(TD_ERR_ARG, "%s: M=%lld / Mk=%lld out of range", fn, (long long)M, (long long)Mk);
  if (M == 0) return TD_OK;
  if (!ws || ws_bytes < (int64_t)carve_attn_layer(nullptr, M, Mk, d, H, self_attention).bytes)
    TD_FAIL(TD_ERR_ARG, "%s: workspace too small", fn);
  return check_pointers(fn, {{"the workspace", ws, kOptionalAligned}});
}
}  // namespace

extern "C" {

int64_t td_t5_attention_layer_workspace_bytes(int64_t M, int64_t Mk, int32_t d, int32_t H, int32_t self_attention) {
  return (int64_t)carve_attn_layer(nullptr, M, Mk, d, H, self_attention != 0).bytes;
}

int32_t td_t5_self_attention_layer_fwd(const void* x, int64_t M, int32_t d, int32_t H, const int32_t* cu_q, int32_t B, int32_t max_len,
                                       const float* ln_w, float eps, const void* w_qkv, const void* wo, const float* bias_by_distance,
                                       int32_t n_dist, void* out, float* rstd, void* qkv, void* o, float* lse, void* ws, int64_t ws_bytes,
                                       td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  const char* fn = "td_t5_self_attention_layer_fwd";
  int rc = attn_layer_check(fn, M, 0, d, H, true, ws, ws_bytes);
  if (rc || M == 0) return rc;
  rc = check_pointers(fn, {{"x", x}, {"ln_w", ln_w}, {"w_qkv", w_qkv}, {"wo", wo}, {"out", out}, {"qkv", qkv, kOptionalAligned},
                           {"o", o, kOptionalAligned}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t inner = kAttnDk * H;
  const AttnLayerWorkspace w = carve_attn_layer(ws, M, 0, d, H, true);
  __nv_bfloat16* qkv_ = qkv ? static_cast<__nv_bfloat16*>(qkv) : w.proj;
  void* o_ = o ? o : w.heads;
  float* rstd_ = rstd ? rstd : w.rstd;
  AttnCall c;  // the attention's own checks, before anything is enqueued
  rc = attn_fwd_check(fn, qkv_, 3 * inner, qkv_ + inner, 3 * inner, qkv_ + 2 * inner, 3 * inner, cu_q, nullptr, B, H, inner, max_len,
                      max_len, M, 1, bias_by_distance, n_dist, o_, inner, lse, c);
  if (rc) return rc;
  rc = rmsnorm_fwd_launch(x, nullptr, 0, ln_w, eps, M, d, w.rows, TD_DTYPE_BF16, rstd_, "sa_norm", st);
  if (rc) return rc;
  rc = gemm_linear(w.rows, M, d, w_qkv, 3 * inner, nullptr, qkv_, w.sk, st, "gemm_sa_qkv");
  if (rc) return rc;
  rc = attn_fwd_run(c, st);
  if (rc) return rc;
  return gemm_residual(o_, M, inner, wo, d, x, out, w.sk, st, "gemm_sa_out");
}

int32_t td_t5_self_attention_layer_bwd(const void* dy, const void* x, const float* rstd, const float* ln_w, const void* qkv, const void* o,
                                       const float* lse, const void* w_qkv, const void* wo, const float* bias_by_distance, int32_t n_dist,
                                       const int32_t* cu_q, int32_t B, int32_t max_len, int64_t M, int32_t d, int32_t H, void* dx, void* dqkv,
                                       void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  const char* fn = "td_t5_self_attention_layer_bwd";
  int rc = attn_layer_check(fn, M, 0, d, H, true, ws, ws_bytes);
  if (rc || M == 0) return rc;
  rc = check_pointers(fn, {{"dy", dy}, {"x", x}, {"rstd", rstd, kNonNull}, {"ln_w", ln_w}, {"qkv", qkv}, {"o", o}, {"lse", lse, kNonNull},
                           {"w_qkv", w_qkv}, {"wo", wo}, {"dx", dx}, {"dqkv", dqkv, kOptionalAligned}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t inner = kAttnDk * H;
  const AttnLayerWorkspace w = carve_attn_layer(ws, M, 0, d, H, true);
  const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(qkv);
  __nv_bfloat16* dq = dqkv ? static_cast<__nv_bfloat16*>(dqkv) : w.proj;
  AttnCall c;
  rc = attn_bwd_check(fn, w.heads, inner, q, 3 * inner, q + inner, 3 * inner, q + 2 * inner, 3 * inner, cu_q, nullptr, B, H, inner, max_len,
                      max_len, M, 1, bias_by_distance, n_dist, o, inner, lse, dq, 3 * inner, dq + inner, 3 * inner, dq + 2 * inner,
                      3 * inner, w.delta, w.delta_bytes, c);
  if (rc) return rc;
  rc = gemm_linear_dx(dy, M, d, wo, inner, w.heads, false, w.sk, st, "gemm_sa_do");
  if (rc) return rc;
  rc = attn_bwd_run(c, st);
  if (rc) return rc;
  rc = gemm_linear_dx(dq, M, 3 * inner, w_qkv, d, w.rows, false, w.sk, st, "gemm_sa_dx");
  if (rc) return rc;
  return residual_norm_bwd_launch(w.rows, x, rstd, ln_w, M, d, dy, dx, "sa_norm_bwd", st);
}

int32_t td_t5_cross_attention_layer_fwd(const void* x, int64_t M, const void* enc, int64_t Mk, int32_t d, int32_t H, const int32_t* cu_q,
                                        const int32_t* cu_k, int32_t B, int32_t max_len_q, int32_t max_len_k, const float* ln_w, float eps,
                                        const void* w_q, const void* w_kv, const void* wo, void* out, float* rstd, void* q, void* kv, void* o,
                                        float* lse, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  const char* fn = "td_t5_cross_attention_layer_fwd";
  int rc = attn_layer_check(fn, M, Mk, d, H, false, ws, ws_bytes);
  if (rc || M == 0) return rc;
  rc = check_pointers(fn, {{"x", x}, {"enc", enc, Mk > 0 ? kNonNullAligned : kOptionalAligned}, {"ln_w", ln_w}, {"w_q", w_q},
                           {"w_kv", w_kv}, {"wo", wo}, {"out", out}, {"q", q, kOptionalAligned}, {"kv", kv, kOptionalAligned},
                           {"o", o, kOptionalAligned}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t inner = kAttnDk * H;
  const AttnLayerWorkspace w = carve_attn_layer(ws, M, Mk, d, H, false);
  void* q_ = q ? q : w.q;
  __nv_bfloat16* kv_ = kv ? static_cast<__nv_bfloat16*>(kv) : w.proj;
  void* o_ = o ? o : w.heads;
  float* rstd_ = rstd ? rstd : w.rstd;
  AttnCall c;
  rc = attn_fwd_check(fn, q_, inner, kv_, 2 * inner, kv_ + inner, 2 * inner, cu_q, cu_k, B, H, inner, max_len_q, max_len_k, M, 0, nullptr,
                      0, o_, inner, lse, c);
  if (rc) return rc;
  rc = rmsnorm_fwd_launch(x, nullptr, 0, ln_w, eps, M, d, w.rows, TD_DTYPE_BF16, rstd_, "ca_norm", st);
  if (rc) return rc;
  rc = gemm_linear(w.rows, M, d, w_q, inner, nullptr, q_, w.sk, st, "gemm_ca_q");
  if (rc) return rc;
  rc = gemm_linear(enc, Mk, d, w_kv, 2 * inner, nullptr, kv_, w.sk, st, "gemm_ca_kv");
  if (rc) return rc;
  rc = attn_fwd_run(c, st);
  if (rc) return rc;
  return gemm_residual(o_, M, inner, wo, d, x, out, w.sk, st, "gemm_ca_out");
}

}  // extern "C"

namespace {
// The two cross-attention backward entries: `accumulate` adds the encoder gradient into d_enc instead of overwriting it.
int cross_attention_layer_bwd(const char* fn, bool accumulate, const void* dy, const void* x, const float* rstd, const float* ln_w,
                              const void* q, const void* kv, const void* o, const float* lse, const void* w_q, const void* w_kv, const void* wo,
                              const int32_t* cu_q, const int32_t* cu_k, int32_t B, int32_t max_len_q, int32_t max_len_k, int64_t M, int64_t Mk,
                              int32_t d, int32_t H, void* dx, float* d_enc, void* ws, int64_t ws_bytes, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  int rc = attn_layer_check(fn, M, Mk, d, H, false, ws, ws_bytes);
  if (rc || M == 0) return rc;
  const PtrRule enc_rule = Mk > 0 ? kNonNullAligned : kOptionalAligned;  // Mk == 0: no key is read, no encoder gradient written
  rc = check_pointers(fn, {{"dy", dy}, {"x", x}, {"rstd", rstd, kNonNull}, {"ln_w", ln_w}, {"q", q}, {"kv", kv, enc_rule}, {"o", o},
                           {"lse", lse, kNonNull}, {"w_q", w_q}, {"w_kv", w_kv}, {"wo", wo}, {"dx", dx}, {"d_enc", d_enc, enc_rule}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t inner = kAttnDk * H;
  const AttnLayerWorkspace w = carve_attn_layer(ws, M, Mk, d, H, false);
  const __nv_bfloat16* k = kv ? static_cast<const __nv_bfloat16*>(kv) : w.proj;  // Mk == 0: no key is read
  AttnCall c;
  rc = attn_bwd_check(fn, w.heads, inner, q, inner, k, 2 * inner, k + inner, 2 * inner, cu_q, cu_k, B, H, inner, max_len_q, max_len_k, M, 0,
                      nullptr, 0, o, inner, lse, w.q, inner, w.proj, 2 * inner, w.proj + inner, 2 * inner, w.delta, w.delta_bytes, c);
  if (rc) return rc;
  rc = gemm_linear_dx(dy, M, d, wo, inner, w.heads, false, w.sk, st, "gemm_ca_do");
  if (rc) return rc;
  rc = attn_bwd_run(c, st);
  if (rc) return rc;
  rc = gemm_linear_dx(w.q, M, inner, w_q, d, w.rows, false, w.sk, st, "gemm_ca_dq");
  if (rc) return rc;
  rc = gemm_linear_dx(w.proj, Mk, 2 * inner, w_kv, d, d_enc, true, w.sk, st, "gemm_ca_denc", accumulate);
  if (rc) return rc;
  return residual_norm_bwd_launch(w.rows, x, rstd, ln_w, M, d, dy, dx, "ca_norm_bwd", st);
}
}  // namespace

extern "C" {

int32_t td_t5_cross_attention_layer_bwd(const void* dy, const void* x, const float* rstd, const float* ln_w, const void* q, const void* kv,
                                        const void* o, const float* lse, const void* w_q, const void* w_kv, const void* wo, const int32_t* cu_q,
                                        const int32_t* cu_k, int32_t B, int32_t max_len_q, int32_t max_len_k, int64_t M, int64_t Mk, int32_t d,
                                        int32_t H, void* dx, float* d_enc, void* ws, int64_t ws_bytes, td_stream_t stream) {
  return cross_attention_layer_bwd("td_t5_cross_attention_layer_bwd", false, dy, x, rstd, ln_w, q, kv, o, lse, w_q, w_kv, wo, cu_q, cu_k, B,
                                   max_len_q, max_len_k, M, Mk, d, H, dx, d_enc, ws, ws_bytes, stream);
}

int32_t td_t5_cross_attention_layer_bwd_accumulate(const void* dy, const void* x, const float* rstd, const float* ln_w, const void* q,
                                                   const void* kv, const void* o, const float* lse, const void* w_q, const void* w_kv,
                                                   const void* wo, const int32_t* cu_q, const int32_t* cu_k, int32_t B, int32_t max_len_q,
                                                   int32_t max_len_k, int64_t M, int64_t Mk, int32_t d, int32_t H, void* dx, float* d_enc,
                                                   void* ws, int64_t ws_bytes, td_stream_t stream) {
  return cross_attention_layer_bwd("td_t5_cross_attention_layer_bwd_accumulate", true, dy, x, rstd, ln_w, q, kv, o, lse, w_q, w_kv, wo, cu_q,
                                   cu_k, B, max_len_q, max_len_k, M, Mk, d, H, dx, d_enc, ws, ws_bytes, stream);
}

// ------------------------------------------------------------------------------------------------ T5 decoder inputs
int32_t td_t5_decoder_inputs(const int64_t* labels, const int32_t* cu_q, int32_t B, int64_t Mq, const void* embed, int64_t V, int32_t d,
                             int64_t decoder_start_token_id, int64_t pad_token_id, void* rows, td_stream_t stream) {
  TD_DEVICE_OR_RETURN();
  const char* fn = "td_t5_decoder_inputs";
  if (B < 0 || Mq < 0 || V <= 0 || d <= 0 || d % 8)
    TD_FAIL(TD_ERR_ARG, "%s: bad sizes (B=%d Mq=%lld V=%lld d=%d; d must be a positive multiple of 8)", fn, B, (long long)Mq, (long long)V, d);
  if (Mq == 0) return TD_OK;
  if (B == 0) TD_FAIL(TD_ERR_ARG, "%s: Mq=%lld rows but no sample", fn, (long long)Mq);
  int rc = check_pointers(fn, {{"labels", labels, kNonNull}, {"cu_q", cu_q, kNonNull}, {"embed", embed}, {"rows", rows}});
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof("t5_decoder_inputs", 4.0 * double(Mq) * d + 8.0 * double(Mq), st);
  PdlConfig l(grid_for_rows(Mq, 8, 8), 256, st);
  TD_CUDA(cudaLaunchKernelEx(&l.cfg, t5_decoder_inputs_kernel, reinterpret_cast<const long long*>(labels), cu_q, B, (long long)Mq,
                             static_cast<const uint4*>(embed), (long long)V, d / 8, (long long)decoder_start_token_id,
                             (long long)pad_token_id, static_cast<uint4*>(rows)));
  return TD_OK;
}

}  // extern "C"
