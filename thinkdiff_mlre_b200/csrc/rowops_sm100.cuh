// HBM-bound kernels of the aligner hot path: ragged pack / pad / mask, fp32->bf16 parameter casts, T5 RMSNorm
// forward and backward, masked MSE and masked cross-entropy (forward + gradient in one pass), and the small
// partial-sum finishers. All of them are byte movers with warp-shuffle reductions: 128-bit global accesses,
// grids sized from the SM count, no shared-memory tiling beyond the CE row stage.
//
// Reference semantics:
//   pack/pad/mask  thinkdiff/datasets/datasets/llava_instruct_dataset_mllama_embed_2.py:101-162
//   T5LayerNorm    transformers modeling_t5.py (imported at thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:24)
//   cross entropy  thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:241-246
#pragma once
#include "ptx_sm100.cuh"

namespace td {

__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  // not volatile, no memory clobber: a read-only (.nc) load is a pure function of its address, so the compiler is
  // free to hoist and batch these ahead of the streaming stores
  asm("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
      : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
      : "l"(p));
  return r;
}
#ifndef TD_ST_VARIANT
#define TD_ST_VARIANT 0
#endif
__device__ __forceinline__ void st_stream(uint4* p, const uint4& v) {
#if TD_ST_VARIANT == 0
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
#elif TD_ST_VARIANT == 1
  *p = v;
#else
  __stcs(p, v);
#endif
}
// 256-bit streaming accesses (sm_100: LDG/STG .256) that are dropped from L2 first: for data touched once per step (optimizer
// state, gradients) next to GEMM operands that should stay resident.
__device__ __forceinline__ void ld256_evict_first(const float* p, float (&r)[8]) {
  uint32_t u[8];
  asm volatile("ld.global.L1::no_allocate.L2::evict_first.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "l"(p));
#pragma unroll
  for (int i = 0; i < 8; ++i) r[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void st256_evict_first(float* p, const float (&r)[8]) {
  asm volatile("st.global.L1::no_allocate.L2::evict_first.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p),
               "r"(__float_as_uint(r[0])), "r"(__float_as_uint(r[1])), "r"(__float_as_uint(r[2])), "r"(__float_as_uint(r[3])),
               "r"(__float_as_uint(r[4])), "r"(__float_as_uint(r[5])), "r"(__float_as_uint(r[6])), "r"(__float_as_uint(r[7]))
               : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------ cu_seqlens
// Exclusive scan of B lengths into int32 cu_seqlens[B+1] (one block; B is a batch size, at most a few thousand).
__global__ void cu_seqlens_kernel(const int* __restrict__ lens, int B, int* __restrict__ cu) {
  grid_dependency_wait();  // launched with programmatic dependent launch: nothing global before this
  grid_launch_dependents();
  __shared__ int warp_tot[32];
  __shared__ int carry;
  if (threadIdx.x == 0) { carry = 0; cu[0] = 0; }
  __syncthreads();
  for (int base = 0; base < B; base += blockDim.x) {
    const int i = base + threadIdx.x;
    int v = i < B ? lens[i] : 0;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[w] = x;
    __syncthreads();
    if (w == 0) {
      int t = lane < (blockDim.x >> 5) ? warp_tot[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += y;
      }
      warp_tot[lane] = t;  // inclusive over warps
    }
    __syncthreads();
    const int before = carry + (w ? warp_tot[w - 1] : 0);
    if (i < B) cu[i + 1] = before + x;
    __syncthreads();
    if (threadIdx.x == 0) carry += warp_tot[(blockDim.x >> 5) - 1];
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------ pack / pad / mask
// One warp moves one destination row per iteration with 128-bit accesses, 8 loads in flight per lane.
//   PADDED = false: dst row r of the packed buffer [M, row] <- sample i = upper_bound(cu, r) - 1, row j = r - cu[i]
//   PADDED = true : dst row r of [B, Lmax, row] <- sample i = r / Lmax, row j = r % Lmax if j < len_i else zeros;
//                   mask[r] = (j < len_i) as int64 (reference mask dtype, ...embed_2.py:118,128)
// Source row = src_row_start[i] + j in the flat source (the un-truncated per-sample embeddings back to back). With a second
// source (src2 != nullptr), a NEGATIVE src_row_start[i] = -(s + 1) means "row s + j of src2": segments of two separate tensors
// are gathered by one launch without concatenating them first (image tokens | text embeddings, BASELINE config 4).
constexpr int kPackMaxStagedSeqs = 2048;  // cu_seqlens / src_row_start are staged in shared memory up to this batch size

template <bool PADDED>
__global__ void __launch_bounds__(256)
pack_rows_kernel(const uint4* __restrict__ src, const long long* __restrict__ src_row_start,
                 const int* __restrict__ cu, int B, long long dst_rows, int Lmax, int vec_per_row,
                 uint4* __restrict__ dst, long long* __restrict__ mask, long long* __restrict__ src_row_out,
                 const uint4* __restrict__ src2 = nullptr) {
  grid_dependency_wait();  // launched with programmatic dependent launch: nothing global before this
  grid_launch_dependents();
  __shared__ int s_cu[kPackMaxStagedSeqs + 1];
  __shared__ long long s_start[kPackMaxStagedSeqs];
  const bool staged = B <= kPackMaxStagedSeqs;
  if (staged) {
    for (int i = threadIdx.x; i <= B; i += blockDim.x) s_cu[i] = cu[i];
    for (int i = threadIdx.x; i < B; i += blockDim.x) s_start[i] = src_row_start[i];
    __syncthreads();
  }
  const int* cu_t = staged ? s_cu : cu;
  const long long* start_t = staged ? s_start : src_row_start;
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long r = warp0; r < dst_rows; r += nwarps) {
    int i, j;
    bool valid = true;
    if constexpr (PADDED) {
      i = int(r / Lmax);
      j = int(r - (long long)i * Lmax);
      valid = j < (cu_t[i + 1] - cu_t[i]);
      if (mask != nullptr && lane == 0) mask[r] = valid ? 1ll : 0ll;
    } else {
      int lo = 0, hi = B;  // largest i with cu[i] <= r
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if ((long long)cu_t[mid] <= r) lo = mid; else hi = mid;
      }
      i = lo;
      j = int(r - (long long)cu_t[i]);
    }
    uint4* d = dst + r * vec_per_row;
    if (valid) {
      long long src_row = start_t[i];
      const uint4* base = src;
      if (src2 != nullptr && src_row < 0) { src_row = -(src_row + 1); base = src2; }
      src_row += j;
      if (src_row_out != nullptr && lane == 0) src_row_out[r] = src_row;  // lets later kernels read sibling tensors unpacked
      const uint4* s = base + src_row * vec_per_row;
      for (int v0 = 0; v0 < vec_per_row; v0 += 256) {
        uint4 t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int v = v0 + u * 32 + lane;
          if (v < vec_per_row) t[u] = ld_stream(s + v);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int v = v0 + u * 32 + lane;
          if (v < vec_per_row) st_stream(d + v, t[u]);
        }
      }
    } else {
      const uint4 z = make_uint4(0, 0, 0, 0);
      for (int v = lane; v < vec_per_row; v += 32) st_stream(d + v, z);
    }
  }
}

// ------------------------------------------------------------------------------------------ casts
__global__ void __launch_bounds__(256)
cast_f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
  const long long n8 = n >> 3;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(src) + 2 * i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(src) + 2 * i + 1);
    reinterpret_cast<uint4*>(dst)[i] =
        make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
  }
  for (long long i = (n8 << 3) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __float2bfloat16_rn(src[i]);
}

// ------------------------------------------------------------------------------------------ T5 RMSNorm forward
// One warp per row. h2 is the bf16 output of Linear2; the variance is taken in fp32 over the bf16 values
// (either summed here, or from the per-N-tile partials the GEMM2 epilogue wrote: ssq_part[P][M]).
//   OUT_BF16 = false: y = g * (h2 * rstd) in fp32            (training: fp32 norm weight)
//   OUT_BF16 = true : y = bf16(g) * bf16(h2 * rstd) -> bf16  (pure-bf16 inference, rounding before the multiply)
constexpr int kNormFwdMaxVec = 16;  // 16 x 32 lanes x 8 bf16 = 4096 columns held in registers per warp

template <bool OUT_BF16>
__global__ void __launch_bounds__(256)
rmsnorm_fwd_kernel(const __nv_bfloat16* __restrict__ h2, const float* __restrict__ ssq_part, int P,
                   const float* __restrict__ g, float eps, int M, int D, void* __restrict__ y_out,
                   float* __restrict__ rstd_out) {
  const int lane = threadIdx.x & 31;
  const int warp0 = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const int nvec = D >> 3;  // uint4 of 8 bf16; nvec <= 32 * kNormFwdMaxVec is enforced on the host
  for (int row = warp0; row < M; row += nwarps) {
    const uint4* hp = reinterpret_cast<const uint4*>(h2 + (long long)row * D);
    // the whole row goes into registers with all loads in flight at once: read from HBM exactly once
    uint4 hu[kNormFwdMaxVec];
#pragma unroll
    for (int k = 0; k < kNormFwdMaxVec; ++k)
      if (lane + 32 * k < nvec) hu[k] = ld_stream(hp + lane + 32 * k);
    float ssq = 0.f;
    if (P > 0) {
      for (int p = lane; p < P; p += 32) ssq += ssq_part[(long long)p * M + row];
    } else {
#pragma unroll
      for (int k = 0; k < kNormFwdMaxVec; ++k) {
        if (lane + 32 * k < nvec) {
          const uint32_t w[4] = {hu[k].x, hu[k].y, hu[k].z, hu[k].w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float a = bf16lo(w[q]), b = bf16hi(w[q]);
            ssq = fmaf(a, a, ssq);
            ssq = fmaf(b, b, ssq);
          }
        }
      }
    }
    ssq = warp_sum(ssq);
    const float rstd = rsqrtf(ssq / float(D) + eps);
    if (lane == 0 && rstd_out != nullptr) rstd_out[row] = rstd;
#pragma unroll
    for (int k = 0; k < kNormFwdMaxVec; ++k) {
      const int v = lane + 32 * k;
      if (v < nvec) {
        const uint32_t w[4] = {hu[k].x, hu[k].y, hu[k].z, hu[k].w};
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(g) + 2 * v);
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(g) + 2 * v + 1);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        float o[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          o[2 * q] = bf16lo(w[q]) * rstd;
          o[2 * q + 1] = bf16hi(w[q]) * rstd;
        }
        if constexpr (OUT_BF16) {
#pragma unroll
          for (int q = 0; q < 8; ++q) o[q] = bf16_round(gg[q]) * bf16_round(o[q]);
          st_stream(reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(y_out) + (long long)row * D) + v,
                    make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]),
                               pack_bf16x2(o[6], o[7])));
        } else {
          uint4* yp = reinterpret_cast<uint4*>(reinterpret_cast<float*>(y_out) + (long long)row * D) + 2 * v;
          st_stream(yp, make_uint4(__float_as_uint(gg[0] * o[0]), __float_as_uint(gg[1] * o[1]),
                                   __float_as_uint(gg[2] * o[2]), __float_as_uint(gg[3] * o[3])));
          st_stream(yp + 1, make_uint4(__float_as_uint(gg[4] * o[4]), __float_as_uint(gg[5] * o[5]),
                                       __float_as_uint(gg[6] * o[6]), __float_as_uint(gg[7] * o[7])));
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ T5 RMSNorm backward
// Thread t of a 512-thread CTA owns columns [8t, 8t+8); the CTA walks its slab of rows R at a time:
//   ghat = g * dy;  s_r = sum_D(ghat * h2)   (block reduction, R rows at once)
//   dh2  = bf16( rstd * ghat - h2 * rstd^3 * s_r / D )
//   dg_part[cta][col] += dy * h2 * rstd;  db2_part[cta][col] += dh2
// Column sums stay in registers and are written once per CTA (deterministic two-level reduction).
// RESIDUAL (a pre-norm sublayer with a frozen weight, T5LayerFF): dh2 = bf16(dres + rstd * ghat - h2 * rstd^3 * s_r / D), the
// gradient that reaches the sublayer's input through the residual branch folded in; no dg / db2 partials.
constexpr int kNormBwdThreads = 512;
constexpr int kNormBwdRows = 2;

template <bool DY_BF16, bool RESIDUAL = false>
__global__ void __launch_bounds__(kNormBwdThreads, 2)
rmsnorm_bwd_kernel(const void* __restrict__ dy_in, const __nv_bfloat16* __restrict__ h2,
                   const float* __restrict__ rstd_in, const float* __restrict__ g, int M, int D, int rows_per_cta,
                   __nv_bfloat16* __restrict__ dh2, float* __restrict__ dg_part, float* __restrict__ db2_part,
                   const __nv_bfloat16* __restrict__ dres = nullptr) {
  constexpr int R = kNormBwdRows;
  __shared__ float red[R][kNormBwdThreads / 32];
  __shared__ float tot[R];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const bool col_ok = t * 8 < D;
  const int row_begin = blockIdx.x * rows_per_cta;
  const int row_end = min(M, row_begin + rows_per_cta);
  float gg[8], adg[8], adb[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) { gg[q] = col_ok ? g[t * 8 + q] : 0.f; adg[q] = 0.f; adb[q] = 0.f; }
  const float inv_d = 1.0f / float(D);

  for (int r0 = row_begin; r0 < row_end; r0 += R) {
    float dyv[R][8], hv[R][8], part[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = r0 + r;
      const bool ok = col_ok && row < row_end;
      uint4 hu = make_uint4(0, 0, 0, 0);
      if (ok) hu = ld_stream(reinterpret_cast<const uint4*>(h2 + (long long)row * D) + t);
      const uint32_t hw[4] = {hu.x, hu.y, hu.z, hu.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) { hv[r][2 * q] = bf16lo(hw[q]); hv[r][2 * q + 1] = bf16hi(hw[q]); }
      if constexpr (DY_BF16) {
        uint4 du = make_uint4(0, 0, 0, 0);
        if (ok) du = ld_stream(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(dy_in) + (long long)row * D) + t);
        const uint32_t dw[4] = {du.x, du.y, du.z, du.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) { dyv[r][2 * q] = bf16lo(dw[q]); dyv[r][2 * q + 1] = bf16hi(dw[q]); }
      } else {
        uint4 d0 = make_uint4(0, 0, 0, 0), d1 = d0;
        if (ok) {
          const uint4* dp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(dy_in) + (long long)row * D) + 2 * t;
          d0 = ld_stream(dp);
          d1 = ld_stream(dp + 1);
        }
        dyv[r][0] = __uint_as_float(d0.x); dyv[r][1] = __uint_as_float(d0.y);
        dyv[r][2] = __uint_as_float(d0.z); dyv[r][3] = __uint_as_float(d0.w);
        dyv[r][4] = __uint_as_float(d1.x); dyv[r][5] = __uint_as_float(d1.y);
        dyv[r][6] = __uint_as_float(d1.z); dyv[r][7] = __uint_as_float(d1.w);
      }
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) s = fmaf(gg[q] * dyv[r][q], hv[r][q], s);
      part[r] = warp_sum(s);
    }
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < R; ++r) red[r][w] = part[r];
    }
    __syncthreads();
    if (w < R) {
      float v = lane < kNormBwdThreads / 32 ? red[w][lane] : 0.f;
      v = warp_sum(v);
      if (lane == 0) tot[w] = v;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = r0 + r;
      if (row < row_end && col_ok) {
        const float rstd = __ldg(rstd_in + row);
        const float c = tot[r] * inv_d * rstd * rstd * rstd;
        float o[8];
        if constexpr (RESIDUAL) {
          float rv[8];
          const uint4 ru = ld_stream(reinterpret_cast<const uint4*>(dres + (long long)row * D) + t);
          const uint32_t rw[4] = {ru.x, ru.y, ru.z, ru.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) { rv[2 * q] = bf16lo(rw[q]); rv[2 * q + 1] = bf16hi(rw[q]); }
#pragma unroll
          for (int q = 0; q < 8; ++q) o[q] = bf16_round(rv[q] + (rstd * gg[q] * dyv[r][q] - hv[r][q] * c));
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            o[q] = bf16_round(rstd * gg[q] * dyv[r][q] - hv[r][q] * c);
            adb[q] += o[q];
            adg[q] = fmaf(dyv[r][q] * hv[r][q], rstd, adg[q]);
          }
        }
        st_stream(reinterpret_cast<uint4*>(dh2 + (long long)row * D) + t,
                  make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]),
                             pack_bf16x2(o[6], o[7])));
      }
    }
    // `tot`/`red` are rewritten only after the next iteration's first __syncthreads(), which every thread
    // reaches after finishing its reads above.
  }
  if (!RESIDUAL && col_ok) {
    float4* pg = reinterpret_cast<float4*>(dg_part + (long long)blockIdx.x * D) + 2 * t;
    float4* pb = reinterpret_cast<float4*>(db2_part + (long long)blockIdx.x * D) + 2 * t;
    pg[0] = make_float4(adg[0], adg[1], adg[2], adg[3]);
    pg[1] = make_float4(adg[4], adg[5], adg[6], adg[7]);
    pb[0] = make_float4(adb[0], adb[1], adb[2], adb[3]);
    pb[1] = make_float4(adb[4], adb[5], adb[6], adb[7]);
  }
}

// ------------------------------------------------------------------------------------------ AdamW (+ bf16 compute copy)
// Decoupled-weight-decay Adam exactly as torch.optim.AdamW (amsgrad=False, maximize=False), the reference optimiser
// (thinkdiff/runners/runner_base.py:122-127):
//   p *= 1 - lr*wd;  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
// One pass also emits the bf16 copy of the parameter that the next forward's GEMMs read (replacing autocast's per-call
// cast), and consumes the gradient straight out of the all-reduced flat bucket. Up to 3 tensors per launch
// (blockIdx.y = segment). 30 B/parameter of HBM traffic.
struct AdamSegment {
  float* p; const float* g; float* m; float* v; __nv_bfloat16* p_bf16; long long n; float weight_decay;
};
// Device-resident control block of one optimizer step (written by step_ctl_kernel): lets GradScaler's inf check / skipped
// step, the unscale factor, the global-norm clip and the bias corrections reach the update kernels without a host sync.
//   torch.amp.GradScaler semantics (thinkdiff/runners/runner_base.py:131-139, tasks/base_task.py:241-258): if any gradient
//   is non-finite the step is skipped for EVERY parameter and the step count does not advance; scale *= backoff, else after
//   growth_interval clean steps scale *= growth.
struct StepCtl {
  int skip;               // 1: non-finite gradient somewhere -> no parameter changes this step
  float grad_mult;        // (1 / loss scale) * clip coefficient, multiplied into every gradient
  float bias_c1;          // 1 - beta1^t
  float sqrt_bias_c2;     // sqrt(1 - beta2^t)
  float step;             // t, the number of applied updates including this one (float: exact up to 2^24)
  float scale;            // current loss scale (the backward's upstream scalar reads this)
  int growth_tracker;     // clean steps since the last scale change
  float grad_norm;        // global gradient norm of this step after unscaling (0 when clipping is off)
};
struct AdamParams {
  AdamSegment seg[3];
  float lr, beta1, beta2, eps, bias_c1, sqrt_bias_c2, grad_scale;
  const StepCtl* ctl;  // optional: overrides bias_c1 / sqrt_bias_c2 / grad_scale and may skip the update
};

__global__ void __launch_bounds__(256)
adamw_kernel(const AdamParams a) {
  const AdamSegment s = a.seg[blockIdx.y];
  const long long n4 = s.n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  float bias_c1 = a.bias_c1, sqrt_bias_c2 = a.sqrt_bias_c2, grad_scale = a.grad_scale;
  if (a.ctl != nullptr) {
    if (a.ctl->skip) return;  // parameters, moments and the bf16 copies all stay as they are
    bias_c1 = a.ctl->bias_c1; sqrt_bias_c2 = a.ctl->sqrt_bias_c2; grad_scale *= a.ctl->grad_mult;
  }
  const float decay = 1.0f - a.lr * s.weight_decay;
  const float step_size = a.lr / bias_c1;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 p = reinterpret_cast<float4*>(s.p)[i];
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(s.g) + i);
    float4 m = reinterpret_cast<float4*>(s.m)[i];
    float4 v = reinterpret_cast<float4*>(s.v)[i];
    float pp[4] = {p.x, p.y, p.z, p.w}, gg[4] = {g4.x, g4.y, g4.z, g4.w}, mm[4] = {m.x, m.y, m.z, m.w}, vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float g = gg[q] * grad_scale;
      pp[q] *= decay;
      mm[q] = a.beta1 * mm[q] + (1.0f - a.beta1) * g;
      vv[q] = a.beta2 * vv[q] + (1.0f - a.beta2) * g * g;
      const float denom = sqrtf(vv[q]) / sqrt_bias_c2 + a.eps;
      pp[q] -= step_size * (mm[q] / denom);
    }
    reinterpret_cast<float4*>(s.p)[i] = make_float4(pp[0], pp[1], pp[2], pp[3]);
    reinterpret_cast<float4*>(s.m)[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
    reinterpret_cast<float4*>(s.v)[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
    if (s.p_bf16 != nullptr)
      reinterpret_cast<uint2*>(s.p_bf16)[i] = make_uint2(pack_bf16x2(pp[0], pp[1]), pack_bf16x2(pp[2], pp[3]));
  }
}

// The same update on 8 parameters per thread and iteration with 256-bit accesses (all sizes and addresses multiples of 32 bytes):
// half the memory instructions, and p / g / m / v are marked evict-first in L2 -- they are not needed again before the next
// optimizer step, while the bf16 copy written last is read by the very next forward GEMM and keeps the default policy.
__global__ void __launch_bounds__(256)
adamw256_kernel(const AdamParams a) {
  const AdamSegment s = a.seg[blockIdx.y];
  const long long n8 = s.n >> 3;
  const long long stride = (long long)gridDim.x * blockDim.x;
  float bias_c1 = a.bias_c1, sqrt_bias_c2 = a.sqrt_bias_c2, grad_scale = a.grad_scale;
  if (a.ctl != nullptr) {
    if (a.ctl->skip) return;
    bias_c1 = a.ctl->bias_c1; sqrt_bias_c2 = a.ctl->sqrt_bias_c2; grad_scale *= a.ctl->grad_mult;
  }
  const float decay = 1.0f - a.lr * s.weight_decay;
  const float step_size = a.lr / bias_c1;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    float pp[8], gg[8], mm[8], vv[8];
    ld256_evict_first(s.p + 8 * i, pp);
    ld256_evict_first(s.g + 8 * i, gg);
    ld256_evict_first(s.m + 8 * i, mm);
    ld256_evict_first(s.v + 8 * i, vv);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float g = gg[q] * grad_scale;
      pp[q] *= decay;
      mm[q] = a.beta1 * mm[q] + (1.0f - a.beta1) * g;
      vv[q] = a.beta2 * vv[q] + (1.0f - a.beta2) * g * g;
      const float denom = sqrtf(vv[q]) / sqrt_bias_c2 + a.eps;
      pp[q] -= step_size * (mm[q] / denom);
    }
    st256_evict_first(s.p + 8 * i, pp);
    st256_evict_first(s.m + 8 * i, mm);
    st256_evict_first(s.v + 8 * i, vv);
    if (s.p_bf16 != nullptr)
      reinterpret_cast<uint4*>(s.p_bf16)[i] = make_uint4(pack_bf16x2(pp[0], pp[1]), pack_bf16x2(pp[2], pp[3]), pack_bf16x2(pp[4], pp[5]),
                                                        pack_bf16x2(pp[6], pp[7]));
  }
}

// One thread: fold this step's gradient statistics into the control block.
//   stats[0] = number of non-finite gradient values seen (summed over ranks), stats[1] = sum of squares of the SCALED gradients
//   (only when clipping). use_scaler = 0: scale stays 1 and nothing is ever skipped (but a clip still applies).
__global__ void step_ctl_kernel(StepCtl* ctl, const float* __restrict__ stats, int use_scaler, float growth, float backoff,
                                int growth_interval, float beta1, float beta2, float max_norm) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float found = stats != nullptr ? stats[0] : 0.f;
  const bool bad = use_scaler && !(found == 0.f);  // NaN counts as found
  const float scale = use_scaler ? ctl->scale : 1.0f;
  const float inv_scale = 1.0f / scale;
  float mult = inv_scale, norm = 0.f;
  if (max_norm > 0.f && stats != nullptr) {
    norm = sqrtf(stats[1]) * inv_scale;
    const float coef = max_norm / (norm + 1e-6f);  // torch.nn.utils.clip_grad_norm_
    mult *= coef < 1.0f ? coef : 1.0f;
    if (!(norm == norm) || norm > 3.0e38f) { /* non-finite norm: torch multiplies by NaN; a scaler would have skipped */ }
  }
  ctl->grad_norm = norm;
  ctl->grad_mult = mult;
  ctl->skip = bad ? 1 : 0;
  if (!bad) {
    const float t = ctl->step + 1.0f;
    ctl->step = t;
    ctl->bias_c1 = float(1.0 - pow((double)beta1, (double)t));
    ctl->sqrt_bias_c2 = float(sqrt(1.0 - pow((double)beta2, (double)t)));
  }
  if (use_scaler) {  // GradScaler.update()
    if (bad) {
      ctl->scale = scale * backoff;
      ctl->growth_tracker = 0;
    } else if (++ctl->growth_tracker == growth_interval) {
      ctl->scale = scale * growth;
      ctl->growth_tracker = 0;
    }
  }
}

// stats[0] += #non-finite, stats[1] += sum of squares over a flat fp32 buffer (grid-stride; one atomic pair per CTA).
__global__ void __launch_bounds__(256)
grad_stats_kernel(const float* __restrict__ g, long long n, float* __restrict__ stats) {
  __shared__ float s_sq[8], s_bad[8];
  float sq = 0.f, bad = 0.f;
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
    const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      sq = fmaf(e[q], e[q], sq);
      bad += (fabsf(e[q]) <= 3.4028234e38f) ? 0.f : 1.f;  // false for inf and NaN
    }
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    sq = fmaf(g[i], g[i], sq);
    bad += (fabsf(g[i]) <= 3.4028234e38f) ? 0.f : 1.f;
  }
  sq = warp_sum(sq); bad = warp_sum(bad);
  if ((threadIdx.x & 31) == 0) { s_sq[threadIdx.x >> 5] = sq; s_bad[threadIdx.x >> 5] = bad; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < 8; ++i) { a += s_sq[i]; b += s_bad[i]; }
    if (b != 0.f) atomicAdd(stats, b);
    atomicAdd(stats + 1, a);
  }
}

// ------------------------------------------------------------------------------------------ fused norm + MSE + norm-backward
// Training against T5 targets never needs y or dy in memory: with y = g * h2 * rstd,
//   diff = y - t;  loss += diff^2;  dy = (2 / (M D)) diff;  then the T5LayerNorm backward of dy, all per row in registers.
// Thread t of a 512-thread CTA owns columns [8t, 8t+8) (so the per-column sums for dg / db2 live in 16 registers); the CTA walks
// its slab of rows two at a time. Each iteration needs ONE block reduction (s_r = sum_D(g dy h2) per row): warps publish their
// partial sums in a parity-double-buffered array, one __syncthreads, every thread adds the 16 partials itself. The loads of the
// next PF iterations are already in flight (packed bf16 in registers) while an iteration computes, so the kernel streams:
// HBM traffic per token is h2 8 KB + target 8 KB (bf16) read, dh2 8 KB written -- instead of the 96 KB of the three separate
// passes (norm fwd 24 KB, MSE 40 KB, norm bwd 32 KB). dh2 / dg / db2 are written for a unit upstream gradient; the backward
// GEMMs and the finisher multiply by the (device-resident) upstream scalar.
constexpr int kNormMseMaxRows = 1024;  // rows whose rstd / target row are staged per block (usually the CTA's whole slab)

template <bool T_BF16>
struct NormMseRow {
  uint4 h;
  uint4 t0;
  uint4 t1;  // second half of the 8 target values when the target is fp32
};

template <bool T_BF16>
__global__ void __launch_bounds__(kNormBwdThreads, 1)
norm_mse_bwd_kernel(const __nv_bfloat16* __restrict__ h2, const float* __restrict__ ssq_part, int P, float eps,
                    const float* __restrict__ g, const void* __restrict__ t_in,
                    const long long* __restrict__ t_row_index, int M, int D, int rows_per_cta, float dy_coef,
                    __nv_bfloat16* __restrict__ dh2, float* __restrict__ dg_part, float* __restrict__ db2_part,
                    float* __restrict__ loss_part) {
  grid_dependency_wait();  // launched with programmatic dependent launch: nothing global before this
  grid_launch_dependents();
  constexpr int R = kNormBwdRows;
  constexpr int PF = T_BF16 ? 2 : 1;  // iterations of loads in flight beyond the one being computed
  constexpr int NB = PF + 1;
  constexpr int NW = kNormBwdThreads / 32;
  static_assert(NW == 16, "the partial-sum butterfly assumes 16 warps");
  __shared__ float red[2][R][NW];
  __shared__ float lred[NW];
  __shared__ float rs_sm[kNormMseMaxRows];
  __shared__ long long ti_sm[kNormMseMaxRows];  // target row of every row of the block (staged: no dependent global loads later)
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const bool col_ok = t * 8 < D;
  const int row_begin = blockIdx.x * rows_per_cta;
  const int row_end = min(M, row_begin + rows_per_cta);
  float gg[8], adg[8], adb[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) { gg[q] = col_ok ? g[t * 8 + q] : 0.f; adg[q] = 0.f; adb[q] = 0.f; }
  const float inv_d = 1.0f / float(D);
  float loss_acc = 0.f;

  for (int b0 = row_begin; b0 < row_end; b0 += kNormMseMaxRows) {
    const int b1 = min(row_end, b0 + kNormMseMaxRows);
    // rstd = rsqrt(mean(h2^2) + eps) from the GEMM2 epilogue's partial sums ssq_part[P][M]: warp w handles rows w, w + 16, ...
    // of the block (lane p reads partial p), so the whole block costs one load round trip
    __syncthreads();  // the previous block's rs_sm / ti_sm / red are no longer read
    for (int i = t; i < b1 - b0; i += kNormBwdThreads)
      ti_sm[i] = t_row_index != nullptr ? __ldg(t_row_index + b0 + i) : (long long)(b0 + i);
    for (int row = b0 + w; row < b1; row += NW) {
      float ssq = 0.f;
      for (int pp = lane; pp < P; pp += 32) ssq += ssq_part[(long long)pp * M + row];
      ssq = warp_sum(ssq);
      if (lane == 0) rs_sm[row - b0] = rsqrtf(ssq / float(D) + eps);
    }
    __syncthreads();

    NormMseRow<T_BF16> buf[NB][R];
    auto issue = [&](NormMseRow<T_BF16> (&dst)[R], int r0) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int row = r0 + r;
        dst[r].h = make_uint4(0, 0, 0, 0); dst[r].t0 = dst[r].h; dst[r].t1 = dst[r].h;
        if (col_ok && row < b1) {
          dst[r].h = ld_stream(reinterpret_cast<const uint4*>(h2 + (long long)row * D) + t);
          const long long trow = ti_sm[row - b0];
          if constexpr (T_BF16) {
            dst[r].t0 = ld_stream(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(t_in) + trow * D) + t);
          } else {
            const uint4* tp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(t_in) + trow * D) + 2 * t;
            dst[r].t0 = ld_stream(tp);
            dst[r].t1 = ld_stream(tp + 1);
          }
        }
      }
    };
#pragma unroll
    for (int u = 0; u < PF; ++u) issue(buf[u], b0 + u * R);

    int it = 0;
    for (int r0 = b0; r0 < b1; r0 += R * NB) {
#pragma unroll
      for (int u = 0; u < NB; ++u) {
        const int rr = r0 + u * R;  // first row of this iteration (uniform across the CTA)
        if (rr < b1) {
          issue(buf[(u + PF) % NB], rr + PF * R);  // refill the buffer consumed in the previous iteration
          // The arithmetic is arranged so that the constant factor of the MSE gradient (dy = dy_coef * diff) is applied once per
          // output instead of once per intermediate -- the kernel is issue-bound (ncu: 57 % issue utilisation, 0.57 of HBM), so
          // every instruction per element counts. With diff = g h rstd - t, u = g h and s' = sum_D(u diff):
          //   dh2 = dy_coef (g (diff rstd) - h s' rstd^3 / D),   dg += dy_coef (diff rstd) h,   loss += diff^2.
          // Rows past the block and columns past D read zeros (h = t = 0, g = 0), so diff is 0 there without a select.
          float df[R][8], hv[R][8], part[R], rs[R];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const int row = rr + r;
            float tv[8];
            const NormMseRow<T_BF16>& in = buf[u][r];
            if constexpr (T_BF16) {
              const uint32_t tw[4] = {in.t0.x, in.t0.y, in.t0.z, in.t0.w};
#pragma unroll
              for (int q = 0; q < 4; ++q) { tv[2 * q] = bf16lo(tw[q]); tv[2 * q + 1] = bf16hi(tw[q]); }
            } else {
              tv[0] = __uint_as_float(in.t0.x); tv[1] = __uint_as_float(in.t0.y); tv[2] = __uint_as_float(in.t0.z); tv[3] = __uint_as_float(in.t0.w);
              tv[4] = __uint_as_float(in.t1.x); tv[5] = __uint_as_float(in.t1.y); tv[6] = __uint_as_float(in.t1.z); tv[7] = __uint_as_float(in.t1.w);
            }
            rs[r] = (row < b1) ? rs_sm[row - b0] : 0.f;
            const uint32_t hw[4] = {in.h.x, in.h.y, in.h.z, in.h.w};
            float sacc = 0.f;
#pragma unroll
            for (int q = 0; q < 4; ++q) { hv[r][2 * q] = bf16lo(hw[q]); hv[r][2 * q + 1] = bf16hi(hw[q]); }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float uq = gg[q] * hv[r][q];
              const float diff = fmaf(uq, rs[r], -tv[q]);
              loss_acc = fmaf(diff, diff, loss_acc);
              sacc = fmaf(uq, diff, sacc);
              df[r][q] = diff;
            }
            part[r] = warp_sum(sacc);
          }
          const int par = it & 1;
          if (lane == 0) {
#pragma unroll
            for (int r = 0; r < R; ++r) red[par][r][w] = part[r];
          }
          __syncthreads();  // the only block barrier of the iteration (the other parity is rewritten one barrier later)
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const int row = rr + r;
            // the 16 warp partials: one shared-memory read per lane, then a 4-step butterfly (same tree in every warp)
            float tot = red[par][r][lane & (NW - 1)];
#pragma unroll
            for (int o = NW / 2; o >= 1; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            if (row < b1 && col_ok) {
              const float rstd = rs[r];
              const float c = tot * inv_d * rstd * rstd * rstd;
              float o[8];
              uint32_t ow[4];
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float t1 = df[r][q] * rstd;
                adg[q] = fmaf(t1, hv[r][q], adg[q]);                      // (dy_coef is applied when the partials are written)
                o[q] = dy_coef * fmaf(gg[q], t1, -hv[r][q] * c);
              }
#pragma unroll
              for (int q = 0; q < 8; q += 2) {  // bf16 rounding through the packed conversion (ALU pipe; the scalar form is an XU-pipe op)
                ow[q >> 1] = bf16_round2(o[q], o[q + 1]);
                adb[q] += o[q];
                adb[q + 1] += o[q + 1];
              }
              st_stream(reinterpret_cast<uint4*>(dh2 + (long long)row * D) + t, make_uint4(ow[0], ow[1], ow[2], ow[3]));
            }
          }
          ++it;
        }
      }
    }
  }
  if (col_ok) {
    float4* pg = reinterpret_cast<float4*>(dg_part + (long long)blockIdx.x * D) + 2 * t;
    float4* pb = reinterpret_cast<float4*>(db2_part + (long long)blockIdx.x * D) + 2 * t;
    pg[0] = make_float4(dy_coef * adg[0], dy_coef * adg[1], dy_coef * adg[2], dy_coef * adg[3]);
    pg[1] = make_float4(dy_coef * adg[4], dy_coef * adg[5], dy_coef * adg[6], dy_coef * adg[7]);
    pb[0] = make_float4(adb[0], adb[1], adb[2], adb[3]);
    pb[1] = make_float4(adb[4], adb[5], adb[6], adb[7]);
  }
  loss_acc = warp_sum(loss_acc);
  if (lane == 0) lred[w] = loss_acc;
  __syncthreads();
  if (t == 0) {
    float tot_loss = 0.f;
    for (int i = 0; i < NW; ++i) tot_loss += lred[i];
    loss_part[blockIdx.x] = tot_loss;
  }
}

// Fixed-order finishers of the two-level reductions, one launch for everything a backward phase needs:
//   job j < njobs : out[n] (+)= scale * (use_scale_ptr ? *scale_ptr : 1) * sum_p part[p][n]  -- column sums (dg, db2 from the norm kernel's per-CTA
//                   partials, db1 from the dh0 GEMM's per-warp-slab partials). One CTA per 32 columns; warp w adds rows
//                   p = w, w + 8, ... (4 independent loads in flight), then the 8 warp sums are combined in warp order.
//   job njobs     : loss = sum(loss_part) / loss_div  (only when loss_out != nullptr)
// Non-finite results bump stats[0] (GradScaler's inf check, see StepCtl).
struct FinishJob { const float* part; float* out; int P; int use_scale_ptr; };
struct FinishParams {
  FinishJob job[3];
  int njobs, N;
  float scale;
  const float* scale_ptr;
  int accumulate;  // 1: out += (gradient accumulation over micro-batches)
  float* stats;    // optional
  const float* loss_part; int loss_P; float* loss_out; float loss_div;
  // peer data parallel: outputs that lie inside [post_base, post_base + post_numel) -- this rank's small-vector bucket -- are ALSO
  // stored at the same offset into post[o], o < n_post: this rank's slot at every rank (the separate posting kernel, folded in)
  float* post[8]; int n_post; const float* post_base; long long post_numel;
};

__global__ void __launch_bounds__(256)
finish_kernel(const FinishParams f) {
  grid_dependency_wait();  // launched with programmatic dependent launch: nothing global before this
  grid_launch_dependents();
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (int(blockIdx.y) == f.njobs) {  // the loss job
    if (blockIdx.x != 0 || f.loss_out == nullptr) return;
    float acc = 0.f;
    for (int i = threadIdx.x; i < f.loss_P; i += blockDim.x) acc += f.loss_part[i];
    acc = warp_sum(acc);
    if (lane == 0) red[w][0] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tot = 0.f;
      for (int i = 0; i < 8; ++i) tot += red[i][0];
      f.loss_out[0] = tot / f.loss_div;
    }
    return;
  }
  const FinishJob j = f.job[blockIdx.y];
  const int col = blockIdx.x * 32 + lane;
  const int N = f.N, P = j.P;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (col < N) {
    int p = w;
    for (; p + 24 < P; p += 32) {
      a0 += j.part[(long long)p * N + col];
      a1 += j.part[(long long)(p + 8) * N + col];
      a2 += j.part[(long long)(p + 16) * N + col];
      a3 += j.part[(long long)(p + 24) * N + col];
    }
    for (; p < P; p += 8) a0 += j.part[(long long)p * N + col];
  }
  red[w][lane] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (w == 0 && col < N) {
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += red[i][lane];
    float v = f.scale * ((j.use_scale_ptr && f.scale_ptr) ? __ldg(f.scale_ptr) : 1.f) * acc;
    if (f.stats != nullptr && !(fabsf(v) <= 3.4028234e38f)) atomicAdd(f.stats, 1.0f);
    if (f.accumulate) v += j.out[col];
    j.out[col] = v;
    if (f.n_post > 0) {
      const long long off = (j.out + col) - f.post_base;
      if (off >= 0 && off < f.post_numel) {
#pragma unroll
        for (int o = 0; o < 8; ++o)
          if (o < f.n_post) f.post[o][off] = v;
      }
    }
  }
}

// Single-job form kept for the module-boundary backward (td_rmsnorm_bwd / td_aligner_bwd).
__global__ void __launch_bounds__(256)
colsum_finish_kernel(const float* __restrict__ part0, float* __restrict__ out0, const float* __restrict__ part1,
                     float* __restrict__ out1, int P, int N, float scale, const float* __restrict__ scale_ptr = nullptr) {
  __shared__ float red[8][33];
  const float* part = blockIdx.y ? part1 : part0;
  float* out = blockIdx.y ? out1 : out0;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + lane;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (col < N) {
    int p = w;
    for (; p + 24 < P; p += 32) {
      a0 += part[(long long)p * N + col];
      a1 += part[(long long)(p + 8) * N + col];
      a2 += part[(long long)(p + 16) * N + col];
      a3 += part[(long long)(p + 24) * N + col];
    }
    for (; p < P; p += 8) a0 += part[(long long)p * N + col];
  }
  red[w][lane] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (w == 0 && col < N) {
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += red[i][lane];
    out[col] = scale * (scale_ptr ? __ldg(scale_ptr) : 1.f) * acc;
  }
}

// ------------------------------------------------------------------------------------------ masked MSE
// loss = sum_valid (y - t)^2 / (n_valid * D);  dy = 2 (y - t) * grad_scale / (n_valid * D) on valid rows, else 0.
// meta[0] = n_valid (float, written by count_valid_kernel or the host), partial sums -> loss_part[grid].
__global__ void count_valid_kernel(const long long* __restrict__ mask, long long n, int ignore_mode,
                                   float* __restrict__ meta) {
  // ignore_mode 0: mask != 0 is valid (attention-mask convention); 1: label != -100 is valid (CE convention)
  __shared__ int wsum[32];
  if (mask == nullptr) {  // no mask: every row counts
    if (threadIdx.x == 0) meta[0] = float(n);
    return;
  }
  int c = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const long long v = mask[i];
    c += ignore_mode ? (v != -100) : (v != 0);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int i = 0; i < (blockDim.x >> 5); ++i) tot += wsum[i];
    meta[0] = float(tot);
  }
}

template <bool Y_BF16, bool T_BF16>
__global__ void __launch_bounds__(256)
masked_mse_kernel(const void* __restrict__ y_in, const void* __restrict__ t_in, const long long* __restrict__ mask,
                  int M, int D, const float* __restrict__ meta, float grad_scale, void* __restrict__ dy_out,
                  float* __restrict__ loss_part) {
  __shared__ float wsum[8];
  const int lane = threadIdx.x & 31;
  const int warp0 = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const int nvec = D >> 3;
  const float n_valid = meta[0];
  const float gs = 2.0f * grad_scale / (n_valid * float(D));
  float acc = 0.f;
  for (int row = warp0; row < M; row += nwarps) {
    const bool valid = mask == nullptr || __ldg(mask + row) != 0;
#pragma unroll 2
    for (int v = lane; v < nvec; v += 32) {
      float yv[8], tv[8];
      if (valid) {
        if constexpr (Y_BF16) {
          const uint4 u = ld_stream(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(y_in) + (long long)row * D) + v);
          const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) { yv[2 * q] = bf16lo(w[q]); yv[2 * q + 1] = bf16hi(w[q]); }
        } else {
          const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(y_in) + (long long)row * D) + 2 * v;
          const uint4 a = ld_stream(p), b = ld_stream(p + 1);
          yv[0] = __uint_as_float(a.x); yv[1] = __uint_as_float(a.y); yv[2] = __uint_as_float(a.z); yv[3] = __uint_as_float(a.w);
          yv[4] = __uint_as_float(b.x); yv[5] = __uint_as_float(b.y); yv[6] = __uint_as_float(b.z); yv[7] = __uint_as_float(b.w);
        }
        if constexpr (T_BF16) {
          const uint4 u = ld_stream(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(t_in) + (long long)row * D) + v);
          const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) { tv[2 * q] = bf16lo(w[q]); tv[2 * q + 1] = bf16hi(w[q]); }
        } else {
          const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(t_in) + (long long)row * D) + 2 * v;
          const uint4 a = ld_stream(p), b = ld_stream(p + 1);
          tv[0] = __uint_as_float(a.x); tv[1] = __uint_as_float(a.y); tv[2] = __uint_as_float(a.z); tv[3] = __uint_as_float(a.w);
          tv[4] = __uint_as_float(b.x); tv[5] = __uint_as_float(b.y); tv[6] = __uint_as_float(b.z); tv[7] = __uint_as_float(b.w);
        }
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) { yv[q] = 0.f; tv[q] = 0.f; }
      }
      float d[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) { d[q] = yv[q] - tv[q]; acc = fmaf(d[q], d[q], acc); d[q] = valid ? d[q] * gs : 0.f; }
      if (dy_out != nullptr) {
        if constexpr (Y_BF16) {
          st_stream(reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(dy_out) + (long long)row * D) + v,
                    make_uint4(pack_bf16x2(d[0], d[1]), pack_bf16x2(d[2], d[3]), pack_bf16x2(d[4], d[5]), pack_bf16x2(d[6], d[7])));
        } else {
          uint4* p = reinterpret_cast<uint4*>(reinterpret_cast<float*>(dy_out) + (long long)row * D) + 2 * v;
          st_stream(p, make_uint4(__float_as_uint(d[0]), __float_as_uint(d[1]), __float_as_uint(d[2]), __float_as_uint(d[3])));
          st_stream(p + 1, make_uint4(__float_as_uint(d[4]), __float_as_uint(d[5]), __float_as_uint(d[6]), __float_as_uint(d[7])));
        }
      }
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) tot += wsum[i];
    loss_part[blockIdx.x] = tot;
  }
}

// loss = sum(part[0..P)) * (use_nd ? 1 / (n_valid * D) : 1 / n_valid); NaN when n_valid == 0 (as torch)
__global__ void loss_finish_kernel(const float* __restrict__ part, int P, const float* __restrict__ meta, float d_or_1,
                                   float* __restrict__ loss, float n_valid_if_no_meta = 0.f) {
  grid_dependency_wait();  // launched with programmatic dependent launch: nothing global before this
  grid_launch_dependents();
  __shared__ float wsum[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < P; i += blockDim.x) acc += part[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) tot += wsum[i];
    loss[0] = tot / ((meta != nullptr ? meta[0] : n_valid_if_no_meta) * d_or_1);
  }
}

// ------------------------------------------------------------------------------------------ masked cross-entropy
// One CTA per logits row. The row is read from HBM exactly once: it is staged in shared memory IN ITS INPUT DTYPE
// (bf16: 64 KB for V = 32128, so three CTAs share an SM) while each thread keeps an online (max, sum-of-exp) pair;
// after one block reduction the gradient is produced from the staged copy:
//   loss_row = logsumexp(z) - z[label];  dz = (softmax(z) - onehot) * grad_scale / n_valid.
// Rows with label == -100 write zeros (ignore_index, ...embed_decoder_2.py:243) and contribute nothing.
constexpr int kCeThreads = 256;

template <bool Z_BF16>
__global__ void __launch_bounds__(kCeThreads, 3)
masked_ce_kernel(const void* __restrict__ z_in, const long long* __restrict__ labels, int V, const float* __restrict__ meta,
                 float grad_scale, void* __restrict__ dz_out, float* __restrict__ row_loss) {
  extern __shared__ uint4 zs[];  // the row, raw: V/8 uint4 (bf16) or V/4 uint4 (fp32)
  __shared__ float red_m[kCeThreads / 32], red_s[kCeThreads / 32];
  __shared__ float bc_m, bc_s;
  constexpr int EPV = Z_BF16 ? 8 : 4;  // elements per 16-byte vector
  const int row = blockIdx.x;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const long long label = labels[row];
  const bool valid = label != -100;
  const int nvec = V / EPV;  // V % 8 == 0 enforced on the host
  const size_t esize = Z_BF16 ? 2 : 4;
  const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(z_in) + (size_t)row * V * esize);
  uint4* dst = dz_out ? reinterpret_cast<uint4*>(reinterpret_cast<char*>(dz_out) + (size_t)row * V * esize) : nullptr;
  if (!valid) {
    if (dst != nullptr) {
      const uint4 z4 = make_uint4(0, 0, 0, 0);
      for (int v = t; v < nvec; v += kCeThreads) st_stream(dst + v, z4);
    }
    if (t == 0) row_loss[row] = 0.f;
    return;
  }
  auto unpack = [](const uint4& u, float* x) {
    if constexpr (Z_BF16) {
      x[0] = bf16lo(u.x); x[1] = bf16hi(u.x); x[2] = bf16lo(u.y); x[3] = bf16hi(u.y);
      x[4] = bf16lo(u.z); x[5] = bf16hi(u.z); x[6] = bf16lo(u.w); x[7] = bf16hi(u.w);
    } else {
      x[0] = __uint_as_float(u.x); x[1] = __uint_as_float(u.y); x[2] = __uint_as_float(u.z); x[3] = __uint_as_float(u.w);
    }
  };
  // pass 1: HBM -> smem, online softmax statistics in base 2 (x * log2e: one FFMA + one MUFU.EX2 per element);
  // 8 independent 16-byte loads in flight per thread
  constexpr float kLog2e = 1.4426950408889634f;
  float m = -INFINITY, ssum = 0.f;  // m is kept in the log2 domain: m = max(x) * log2e
  constexpr int U = 8;
  for (int v0 = t; v0 < nvec; v0 += kCeThreads * U) {
    uint4 u[U];
#pragma unroll
    for (int k = 0; k < U; ++k)
      if (v0 + k * kCeThreads < nvec) u[k] = ld_stream(src + v0 + k * kCeThreads);
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int v = v0 + k * kCeThreads;
      if (v >= nvec) break;
      zs[v] = u[k];
      float x[8];
      unpack(u[k], x);
      float vm = x[0];
#pragma unroll
      for (int q = 1; q < EPV; ++q) vm = fmaxf(vm, x[q]);
      vm *= kLog2e;
      if (vm > m) { ssum *= exp2f(m - vm); m = vm; }
#pragma unroll
      for (int q = 0; q < EPV; ++q) ssum += exp2f(fmaf(x[q], kLog2e, -m));
    }
  }
  // block reduction of (m, ssum)
  float wm = warp_max(m);
  ssum = (m == -INFINITY) ? 0.f : ssum * exp2f(m - wm);  // idle threads (m = -inf) contribute nothing
  ssum = warp_sum(ssum);
  if (lane == 0) { red_m[w] = wm; red_s[w] = ssum; }
  __syncthreads();
  if (w == 0) {
    float mm = lane < kCeThreads / 32 ? red_m[lane] : -INFINITY;
    float sv = lane < kCeThreads / 32 ? red_s[lane] : 0.f;
    const float bm = warp_max(mm);
    sv = (mm == -INFINITY) ? 0.f : sv * exp2f(mm - bm);
    sv = warp_sum(sv);
    if (lane == 0) { bc_m = bm; bc_s = sv; }
  }
  __syncthreads();
  const float mx = bc_m, sum = bc_s;
  if (t == 0) {
    float zl = __int_as_float(0x7fc00000);
    if (label >= 0 && label < V) {
      if constexpr (Z_BF16) zl = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(zs)[label]);
      else zl = reinterpret_cast<const float*>(zs)[label];
    }
    row_loss[row] = (logf(sum) + mx * 0.6931471805599453f) - zl;  // mx is in the log2 domain
  }
  if (dst == nullptr) return;
  // pass 2: gradient from the staged row. softmax * gs = exp2(x * log2e - mx + log2(gs / sum)): one FFMA + one MUFU per
  // element; the "- onehot" correction is applied once, by the thread that owns the label's vector.
  const float gs = grad_scale / meta[0];
  const float shift = -mx + log2f(fabsf(gs) / sum);
  const float sgn = gs < 0.f ? -1.f : 1.f;
  const int label_vec = (label >= 0 && label < V) ? int(label) / EPV : -1;
  for (int v = t; v < nvec; v += kCeThreads) {
    float x[8];
    unpack(zs[v], x);
#pragma unroll
    for (int q = 0; q < EPV; ++q) x[q] = sgn * exp2f(fmaf(x[q], kLog2e, shift));
    if (v == label_vec) x[int(label) - v * EPV] -= gs;
    if constexpr (Z_BF16)
      st_stream(dst + v, make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7])));
    else
      st_stream(dst + v, make_uint4(__float_as_uint(x[0]), __float_as_uint(x[1]), __float_as_uint(x[2]), __float_as_uint(x[3])));
  }
}

}  // namespace td
