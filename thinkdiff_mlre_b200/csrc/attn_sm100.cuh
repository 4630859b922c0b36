// T5 attention core on packed rows (SURVEY section 8 f-1), forward and backward, on tcgen05:
//
//   cross : O[i] = softmax_j( q_i . k_j )                         j < L_b            (decoder rows attend to the aligner rows)
//   self  : O[i] = softmax_j( q_i . k_j + bias[h, min(i - j, n_dist - 1)] )   j <= i    (causal, positions from the sample's start)
//
// T5 rules: no 1/sqrt(d_kv) scaling, softmax in fp32, d_kv = 64. Sample b's queries are rows cu_q[b]..cu_q[b+1] of Q, its keys /
// values rows cu_k[b]..cu_k[b+1] of K / V; head h is columns [64 h, 64 h + 64) of every row (row pitches are free, so Q/K/V may
// be column slices of one fused projection output).
//
// Layout of every operand tile in shared memory: 128 rows x 64 bf16 = 128 rows of 128 bytes with the 128-byte swizzle (16-byte
// piece c of row r at r * 128 + ((c ^ (r & 7)) << 4)). That one layout serves both operand kinds of the tensor core: read as
// K-major it is [rows, 64] with the contraction over the 64 columns (Q . K^T, dO . V^T); read as MN-major it is [K = 128 rows, N = 64]
// with the contraction over the rows (P . V, dS . K, P^T . dO, dS^T . Q) -- the descriptor kind the weight-gradient GEMMs use.
// The 128 x 128 probability / score-gradient tiles the softmax threads write are two such tiles side by side (keys 0-63, 64-127).
//
// Tiles are loaded with cp.async, 16 bytes per thread and row-predicated: rows past the sample's end are zero-filled instead of
// read, so a partial tile never sees the neighbouring sample and masked keys contribute exact zeros to P . V. Every store is
// row-predicated too (a whole-tile store would overwrite the next sample's rows).
//
// Kernels (128 threads = one thread per tile row; thread 0 issues the MMAs):
//   t5_attn_fwd_kernel     one CTA per (128-query tile, head, sample), loop over key tiles: S = Q.K^T -> TMEM (128 cols),
//                          row max / exp / sum by the owning thread, P (bf16) -> smem, P.V -> TMEM (64 cols), O = O * alpha + P.V
//                          kept in registers (the online-softmax correction). Writes O (bf16) and LSE (fp32, natural log).
//   t5_attn_delta_kernel   Delta[h, i] = sum_d dO[i, h, d] * O[i, h, d]
//   t5_attn_dkdv_kernel    one CTA per (128-key tile, head, sample), loop over query tiles: S^T = K.Q^T, dP^T = V.dO^T (TMEM),
//                          P^T = exp(S^T + bias - LSE), dS^T = P^T (dP^T - Delta) (bf16 -> smem), dV += P^T.dO, dK += dS^T.Q (TMEM)
//   t5_attn_dq_kernel      one CTA per (128-query tile, head, sample), loop over key tiles: S = Q.K^T, dP = dO.V^T (TMEM),
//                          dS -> smem, dQ += dS.K (product in TMEM, sum in registers)
// Every output element is written by exactly one CTA: deterministic, no atomics. CTAs past a sample's end exit at once.
#pragma once
#include "ptx_sm100.cuh"

namespace td {

constexpr int kAttnTile = 128;                       // rows per query / key tile = TMEM lanes = UMMA M
constexpr int kAttnDk = 64;                          // d_kv
constexpr int kAttnThreads = 128;
constexpr int kAttnTileBytes = kAttnTile * kAttnDk * 2;  // 16 KB
constexpr int kAttnMaxDist = 4096;                   // bias-table entries staged in shared memory
constexpr float kLog2e = 1.4426950408889634f;

struct AttnParams {
  const __nv_bfloat16 *q, *k, *v, *o, *dout;
  long long ldq, ldk, ldv, ldo, lddo;
  const int *cu_q, *cu_k;
  const float* bias;  // [H, n_dist] (self-attention) or nullptr (cross)
  int n_dist, H;
  long long Mq;
  float* lse;          // [H, Mq]
  float* delta;        // [H, Mq]
  __nv_bfloat16 *out, *dq, *dk, *dv;
  long long ld_out, lddq, lddk, lddv;
};

// Shared-memory plan of each kernel (byte offsets from a 1024-aligned base).
struct AttnFwdSmem {
  static constexpr int kQ = 0, kK = kQ + kAttnTileBytes, kV = kK + kAttnTileBytes, kP = kV + kAttnTileBytes;
  static constexpr int kBar = kP + 2 * kAttnTileBytes, kBias = kBar + 64;
};
struct AttnDkdvSmem {
  static constexpr int kK = 0, kV = kK + kAttnTileBytes, kQ = kV + kAttnTileBytes, kDo = kQ + kAttnTileBytes;
  static constexpr int kPt = kDo + kAttnTileBytes, kDst = kPt + 2 * kAttnTileBytes;
  static constexpr int kLse = kDst + 2 * kAttnTileBytes, kDelta = kLse + 4 * kAttnTile, kBar = kDelta + 4 * kAttnTile, kBias = kBar + 64;
};
struct AttnDqSmem {
  static constexpr int kQ = 0, kDo = kQ + kAttnTileBytes, kK = kDo + kAttnTileBytes, kV = kK + kAttnTileBytes;
  static constexpr int kDs = kV + kAttnTileBytes, kBar = kDs + 2 * kAttnTileBytes, kBias = kBar + 64;
};
// dynamic shared memory of a launch: the plan, the bias table and the alignment slack
__host__ __device__ constexpr int attn_smem_bytes(int bias_off, int n_dist) { return bias_off + 4 * n_dist + 1024; }

__device__ __forceinline__ uint32_t attn_sw128(int r, int c) { return uint32_t(r * 128 + ((c ^ (r & 7)) << 4)); }

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, bool valid) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Rows [row0, row0 + 128) of head `h` into a swizzled tile; rows >= n_valid are zero-filled (never read).
__device__ __forceinline__ void attn_load_tile(uint8_t* tile, const __nv_bfloat16* base, long long ld, long long row0, int n_valid,
                                               int h, int tid) {
  const uint32_t s = smem_u32(tile);
#pragma unroll
  for (int it = 0; it < kAttnTile * 8 / kAttnThreads; ++it) {
    const int idx = it * kAttnThreads + tid;
    const int r = idx >> 3, c = idx & 7;
    const bool ok = r < n_valid;
    const __nv_bfloat16* src = ok ? base + (row0 + r) * ld + h * kAttnDk + c * 8 : base;
    cp_async16_zfill(s + attn_sw128(r, c), src, ok);
  }
}

// Shared-memory descriptors. K-major [rows, 64]: the k-th 16-column slice starts 32 bytes further. MN-major [128 k-rows, 64]: the
// k-th 16-row slice starts 2048 bytes further (LBO would be the next 64-column block; N = 64 has none).
__device__ __forceinline__ uint64_t attn_desc_kmajor(uint32_t tile, int k) { return make_smem_desc_sw128(tile + k * 32, 16, 1024); }
__device__ __forceinline__ uint64_t attn_desc_mnmajor(uint32_t tile, int k) { return make_smem_desc_sw128(tile + k * 2048, 8192, 1024); }
// A 128 x 128 K-major operand stored as two [128, 64] tiles: slice k (of 8) of the 128-long contraction.
__device__ __forceinline__ uint64_t attn_desc_kmajor_wide(uint32_t tile2, int k) {
  return attn_desc_kmajor(tile2 + (k >> 2) * kAttnTileBytes, k & 3);
}

constexpr uint32_t kIdescSS = make_idesc_bf16(kAttnTile, kAttnTile, false, false);  // [128 x 64] . [128 x 64]^T -> 128 x 128
constexpr uint32_t kIdescPV = make_idesc_bf16(kAttnTile, kAttnDk, false, true);      // [128 x 128] . [128 k-rows x 64] -> 128 x 64

// 128 x 128 (A) by 128 x 64 (B, MN-major) into TMEM columns [col, col + 64)
__device__ __forceinline__ void attn_mma_pv(uint32_t tmem_d, uint32_t a_tile2, uint32_t b_tile, bool accumulate) {
#pragma unroll
  for (int k = 0; k < kAttnTile / 16; ++k)
    umma_bf16<1>(tmem_d, attn_desc_kmajor_wide(a_tile2, k), attn_desc_mnmajor(b_tile, k), kIdescPV, (accumulate || k > 0) ? 1u : 0u);
}
// 128 x 64 (A) by 128 x 64 (B), both K-major, into TMEM columns [col, col + 128)
__device__ __forceinline__ void attn_mma_ss(uint32_t tmem_d, uint32_t a_tile, uint32_t b_tile) {
#pragma unroll
  for (int k = 0; k < kAttnDk / 16; ++k)
    umma_bf16<1>(tmem_d, attn_desc_kmajor(a_tile, k), attn_desc_kmajor(b_tile, k), kIdescSS, k > 0 ? 1u : 0u);
}

// 32 bf16 values (one TMEM chunk of a thread's row) into the two-tile 128 x 128 operand at columns [32 c, 32 c + 32).
__device__ __forceinline__ void attn_store_row_chunk(uint8_t* tile2, int row, int c, const float* x) {
  uint8_t* t = tile2 + (c >> 1) * kAttnTileBytes;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float* y = x + g * 8;
    *reinterpret_cast<uint4*>(t + attn_sw128(row, (c & 1) * 4 + g)) =
        make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
  }
}

// 64 fp32 values -> one bf16 head row in global memory (row-predicated by the caller).
__device__ __forceinline__ void attn_store_row(__nv_bfloat16* dst, const float* x, float scale) {
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    const float* y = x + g * 8;
    reinterpret_cast<uint4*>(dst)[g] = make_uint4(pack_bf16x2(y[0] * scale, y[1] * scale), pack_bf16x2(y[2] * scale, y[3] * scale),
                                                  pack_bf16x2(y[4] * scale, y[5] * scale), pack_bf16x2(y[6] * scale, y[7] * scale));
  }
}

// All threads: wait for the MMAs committed to `bar`, then make their TMEM results visible.
__device__ __forceinline__ void attn_wait_mma(uint64_t* bar, uint32_t parity) {
  mbar_wait(bar, parity);
  tc_fence_after();
}
// All threads: hand the smem they wrote (cp.async tiles or st.shared operands) and the TMEM they read over to the MMA issuer.
__device__ __forceinline__ void attn_sync_for_mma() {
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
}

__device__ __forceinline__ uint8_t* attn_smem_base() {
  extern __shared__ uint8_t attn_smem_raw[];
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(attn_smem_raw) + 1023) & ~uintptr_t(1023));
}

// Common prologue: TMEM allocation (warp 0), two mbarriers, the head's bias table. Returns the TMEM base.
__device__ __forceinline__ uint32_t attn_prologue(uint8_t* smem, int bar_off, int bias_off, const AttnParams& p, int h, int tid,
                                                  uint32_t tmem_cols) {
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + bar_off);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + bar_off + 32);
  if (tid < 32) {
    tmem_alloc<1>(tmem_slot, tmem_cols);
    tmem_relinquish<1>();
  }
  if (tid == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    fence_mbar_init();
  }
  if (p.bias != nullptr) {
    float* bias_s = reinterpret_cast<float*>(smem + bias_off);
    for (int n = tid; n < p.n_dist; n += kAttnThreads) bias_s[n] = __ldg(p.bias + (size_t)h * p.n_dist + n);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return *tmem_slot;
}
__device__ __forceinline__ void attn_epilogue(uint32_t tmem, uint32_t tmem_cols, int tid) {
  tc_fence_before();
  __syncthreads();
  if (tid < 32) {
    tc_fence_after();
    tmem_dealloc<1>(tmem, tmem_cols);
  }
}

// Score of (query position i, key position j) from the raw product; -inf when masked.
__device__ __forceinline__ float attn_score(float s, int i, int j, int L, bool causal, const float* bias_s, int n_dist) {
  if (j >= L) return -INFINITY;
  if (causal) {
    if (j > i) return -INFINITY;
    const int n = i - j;
    s += bias_s[n < n_dist ? n : n_dist - 1];
  }
  return s;
}

// ------------------------------------------------------------------------------------------------ forward
template <bool CAUSAL>
__global__ void __launch_bounds__(kAttnThreads) t5_attn_fwd_kernel(const AttnParams p) {
  using S = AttnFwdSmem;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = __ldg(p.cu_q + b), T = __ldg(p.cu_q + b + 1) - q0;
  if (qt * kAttnTile >= T) return;
  const int k0 = __ldg(p.cu_k + b), L = __ldg(p.cu_k + b + 1) - k0;
  const int tid = threadIdx.x, warp = tid >> 5;
  uint8_t* smem = attn_smem_base();
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::kBar);
  const float* bias_s = reinterpret_cast<const float*>(smem + S::kBias);
  const uint32_t tmem = attn_prologue(smem, S::kBar, S::kBias, p, h, tid, 256);
  const uint32_t s_q = smem_u32(smem + S::kQ), s_k = smem_u32(smem + S::kK), s_v = smem_u32(smem + S::kV), s_p = smem_u32(smem + S::kP);
  const uint32_t trow = tmem + (uint32_t(warp * 32) << 16);

  attn_load_tile(smem + S::kQ, p.q, p.ldq, q0 + qt * kAttnTile, T - qt * kAttnTile, h, tid);
  const int key_tiles = (L + kAttnTile - 1) / kAttnTile;
  const int n_kt = CAUSAL ? (qt + 1 < key_tiles ? qt + 1 : key_tiles) : key_tiles;
  const int i = qt * kAttnTile + tid;  // this thread's query position in the sample
  float o[kAttnDk];
#pragma unroll
  for (int d = 0; d < kAttnDk; ++d) o[d] = 0.f;
  float m = -INFINITY, l = 0.f;

#pragma unroll 1
  for (int kt = 0; kt < n_kt; ++kt) {
    attn_load_tile(smem + S::kK, p.k, p.ldk, k0 + kt * kAttnTile, L - kt * kAttnTile, h, tid);
    attn_load_tile(smem + S::kV, p.v, p.ldv, k0 + kt * kAttnTile, L - kt * kAttnTile, h, tid);
    cp_async_wait_all();
    attn_sync_for_mma();
    if (tid == 0) {
      tc_fence_after();
      attn_mma_ss(tmem, s_q, s_k);
      umma_commit<1>(&bar[0]);
    }
    attn_wait_mma(&bar[0], kt & 1);
    const int j0 = kt * kAttnTile;
    float mt = -INFINITY;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(trow + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) mt = fmaxf(mt, attn_score(__uint_as_float(v[jj]), i, j0 + c * 32 + jj, L, CAUSAL, bias_s, p.n_dist));
    }
    const float m_new = fmaxf(m, mt);
    const float m_ref = m_new == -INFINITY ? 0.f : m_new;  // a row with nothing visible yet keeps p = 0
    const float alpha = ex2_approx((m - m_ref) * kLog2e);
    const float mref2 = m_ref * kLog2e;
    float lt = 0.f;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(trow + c * 32, v);
      tmem_ld_wait();
      float pr[32];
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) {
        const float s = attn_score(__uint_as_float(v[jj]), i, j0 + c * 32 + jj, L, CAUSAL, bias_s, p.n_dist);
        pr[jj] = ex2_approx(fmaf(s, kLog2e, -mref2));
        lt += pr[jj];
      }
      attn_store_row_chunk(smem + S::kP, tid, c, pr);
    }
    l = l * alpha + lt;
    m = m_new;
    attn_sync_for_mma();
    if (tid == 0) {
      tc_fence_after();
      attn_mma_pv(tmem + kAttnTile, s_p, s_v, false);
      umma_commit<1>(&bar[1]);
    }
    attn_wait_mma(&bar[1], kt & 1);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(trow + kAttnTile + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int d = 0; d < 32; ++d) o[c * 32 + d] = fmaf(o[c * 32 + d], alpha, __uint_as_float(v[d]));
    }
  }
  if (i < T) {
    const float inv = l > 0.f ? 1.f / l : 0.f;  // L_b = 0: O = 0
    attn_store_row(p.out + (q0 + i) * p.ld_out + h * kAttnDk, o, inv);
    if (p.lse != nullptr) p.lse[(size_t)h * p.Mq + q0 + i] = l > 0.f ? m + logf(l) : -INFINITY;
  }
  attn_epilogue(tmem, 256, tid);
}

// ------------------------------------------------------------------------------------------------ backward
// Delta[h, r] = sum_d dO[r, 64 h + d] * O[r, 64 h + d] for every row r < Mq: 8 threads per (row, head), 16 bytes each.
__global__ void __launch_bounds__(256) t5_attn_delta_kernel(const AttnParams p) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long pair = gid >> 3;
  const int part = int(gid & 7);
  const bool ok = pair < p.Mq * p.H;
  const long long r = ok ? pair / p.H : 0;
  const int h = ok ? int(pair - r * p.H) : 0;
  float acc = 0.f;
  if (ok) {
    const uint4 a = *reinterpret_cast<const uint4*>(p.o + r * p.ldo + h * kAttnDk + part * 8);
    const uint4 g = *reinterpret_cast<const uint4*>(p.dout + r * p.lddo + h * kAttnDk + part * 8);
    acc = bf16lo(a.x) * bf16lo(g.x) + bf16hi(a.x) * bf16hi(g.x) + bf16lo(a.y) * bf16lo(g.y) + bf16hi(a.y) * bf16hi(g.y) +
          bf16lo(a.z) * bf16lo(g.z) + bf16hi(a.z) * bf16hi(g.z) + bf16lo(a.w) * bf16lo(g.w) + bf16hi(a.w) * bf16hi(g.w);
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  if (ok && part == 0) p.delta[(size_t)h * p.Mq + r] = acc;
}

template <bool CAUSAL>
__global__ void __launch_bounds__(kAttnThreads, 1) t5_attn_dkdv_kernel(const AttnParams p) {
  using S = AttnDkdvSmem;
  const int kt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int k0 = __ldg(p.cu_k + b), L = __ldg(p.cu_k + b + 1) - k0;
  if (kt * kAttnTile >= L) return;
  const int q0 = __ldg(p.cu_q + b), T = __ldg(p.cu_q + b + 1) - q0;
  const int tid = threadIdx.x, warp = tid >> 5;
  uint8_t* smem = attn_smem_base();
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::kBar);
  const float* bias_s = reinterpret_cast<const float*>(smem + S::kBias);
  float* lse_s = reinterpret_cast<float*>(smem + S::kLse);
  float* delta_s = reinterpret_cast<float*>(smem + S::kDelta);
  // TMEM: S^T [0, 128), dP^T [128, 256), dV [256, 320), dK [320, 384)
  const uint32_t tmem = attn_prologue(smem, S::kBar, S::kBias, p, h, tid, 512);
  const uint32_t s_k = smem_u32(smem + S::kK), s_v = smem_u32(smem + S::kV), s_q = smem_u32(smem + S::kQ), s_do = smem_u32(smem + S::kDo);
  const uint32_t s_pt = smem_u32(smem + S::kPt), s_dst = smem_u32(smem + S::kDst);
  const uint32_t trow = tmem + (uint32_t(warp * 32) << 16);

  attn_load_tile(smem + S::kK, p.k, p.ldk, k0 + kt * kAttnTile, L - kt * kAttnTile, h, tid);
  attn_load_tile(smem + S::kV, p.v, p.ldv, k0 + kt * kAttnTile, L - kt * kAttnTile, h, tid);
  const int j = kt * kAttnTile + tid;  // this thread's key position
  const int qt0 = CAUSAL ? kt : 0;
  const int n_qt = (T + kAttnTile - 1) / kAttnTile;
  int it = 0;
#pragma unroll 1
  for (int qt = qt0; qt < n_qt; ++qt, ++it) {
    attn_load_tile(smem + S::kQ, p.q, p.ldq, q0 + qt * kAttnTile, T - qt * kAttnTile, h, tid);
    attn_load_tile(smem + S::kDo, p.dout, p.lddo, q0 + qt * kAttnTile, T - qt * kAttnTile, h, tid);
    {
      const int iq = qt * kAttnTile + tid;
      lse_s[tid] = iq < T ? __ldg(p.lse + (size_t)h * p.Mq + q0 + iq) * kLog2e : 0.f;
      delta_s[tid] = iq < T ? __ldg(p.delta + (size_t)h * p.Mq + q0 + iq) : 0.f;
    }
    cp_async_wait_all();
    attn_sync_for_mma();
    if (tid == 0) {
      tc_fence_after();
      attn_mma_ss(tmem, s_k, s_q);               // S^T = K . Q^T
      attn_mma_ss(tmem + kAttnTile, s_v, s_do);  // dP^T = V . dO^T
      umma_commit<1>(&bar[0]);
    }
    attn_wait_mma(&bar[0], it & 1);
    const int i0 = qt * kAttnTile;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t sv[32], dv[32];
      tmem_ld_32x32(trow + c * 32, sv);
      tmem_ld_32x32(trow + kAttnTile + c * 32, dv);
      tmem_ld_wait();
      float pr[32], ds[32];
#pragma unroll
      for (int ii = 0; ii < 32; ++ii) {
        const int i = i0 + c * 32 + ii;
        const float s = attn_score(__uint_as_float(sv[ii]), i, j, L, CAUSAL, bias_s, p.n_dist);
        const bool vis = i < T && s != -INFINITY;
        const float pv = vis ? ex2_approx(fmaf(s, kLog2e, -lse_s[c * 32 + ii])) : 0.f;
        pr[ii] = pv;
        ds[ii] = pv * (__uint_as_float(dv[ii]) - delta_s[c * 32 + ii]);
      }
      attn_store_row_chunk(smem + S::kPt, tid, c, pr);
      attn_store_row_chunk(smem + S::kDst, tid, c, ds);
    }
    attn_sync_for_mma();
    if (tid == 0) {
      tc_fence_after();
      attn_mma_pv(tmem + 2 * kAttnTile, s_pt, s_do, it > 0);                // dV += P^T . dO
      attn_mma_pv(tmem + 2 * kAttnTile + kAttnDk, s_dst, s_q, it > 0);      // dK += dS^T . Q
      umma_commit<1>(&bar[1]);
    }
    attn_wait_mma(&bar[1], it & 1);  // Q / dO / P^T / dS^T are reused by the next query tile
  }
  // (the TMEM loads are warp-collective: every lane loads, only rows of the sample store)
#pragma unroll 1
  for (int t = 0; t < 2; ++t) {
    float acc[kAttnDk];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(trow + 2 * kAttnTile + t * kAttnDk + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int d = 0; d < 32; ++d) acc[c * 32 + d] = it > 0 ? __uint_as_float(v[d]) : 0.f;  // it == 0: no query sees these keys
    }
    if (j < L) attn_store_row(t == 0 ? p.dv + (k0 + j) * p.lddv + h * kAttnDk : p.dk + (k0 + j) * p.lddk + h * kAttnDk, acc, 1.f);
  }
  attn_epilogue(tmem, 512, tid);
}

template <bool CAUSAL>
__global__ void __launch_bounds__(kAttnThreads) t5_attn_dq_kernel(const AttnParams p) {
  using S = AttnDqSmem;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = __ldg(p.cu_q + b), T = __ldg(p.cu_q + b + 1) - q0;
  if (qt * kAttnTile >= T) return;
  const int k0 = __ldg(p.cu_k + b), L = __ldg(p.cu_k + b + 1) - k0;
  const int tid = threadIdx.x, warp = tid >> 5;
  uint8_t* smem = attn_smem_base();
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::kBar);
  const float* bias_s = reinterpret_cast<const float*>(smem + S::kBias);
  // TMEM: S [0, 128) (its first 64 columns take the dS . K product once S has been read), dP [128, 256)
  const uint32_t tmem = attn_prologue(smem, S::kBar, S::kBias, p, h, tid, 256);
  const uint32_t s_q = smem_u32(smem + S::kQ), s_do = smem_u32(smem + S::kDo), s_k = smem_u32(smem + S::kK), s_v = smem_u32(smem + S::kV);
  const uint32_t s_ds = smem_u32(smem + S::kDs);
  const uint32_t trow = tmem + (uint32_t(warp * 32) << 16);

  attn_load_tile(smem + S::kQ, p.q, p.ldq, q0 + qt * kAttnTile, T - qt * kAttnTile, h, tid);
  attn_load_tile(smem + S::kDo, p.dout, p.lddo, q0 + qt * kAttnTile, T - qt * kAttnTile, h, tid);
  const int i = qt * kAttnTile + tid;
  const float lse2 = i < T ? __ldg(p.lse + (size_t)h * p.Mq + q0 + i) * kLog2e : 0.f;
  const float delta = i < T ? __ldg(p.delta + (size_t)h * p.Mq + q0 + i) : 0.f;
  const int key_tiles = (L + kAttnTile - 1) / kAttnTile;
  const int n_kt = CAUSAL ? (qt + 1 < key_tiles ? qt + 1 : key_tiles) : key_tiles;
  float dq[kAttnDk];
#pragma unroll
  for (int d = 0; d < kAttnDk; ++d) dq[d] = 0.f;

#pragma unroll 1
  for (int kt = 0; kt < n_kt; ++kt) {
    attn_load_tile(smem + S::kK, p.k, p.ldk, k0 + kt * kAttnTile, L - kt * kAttnTile, h, tid);
    attn_load_tile(smem + S::kV, p.v, p.ldv, k0 + kt * kAttnTile, L - kt * kAttnTile, h, tid);
    cp_async_wait_all();
    attn_sync_for_mma();
    if (tid == 0) {
      tc_fence_after();
      attn_mma_ss(tmem, s_q, s_k);                // S = Q . K^T
      attn_mma_ss(tmem + kAttnTile, s_do, s_v);   // dP = dO . V^T
      umma_commit<1>(&bar[0]);
    }
    attn_wait_mma(&bar[0], kt & 1);
    const int j0 = kt * kAttnTile;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t sv[32], dv[32];
      tmem_ld_32x32(trow + c * 32, sv);
      tmem_ld_32x32(trow + kAttnTile + c * 32, dv);
      tmem_ld_wait();
      float ds[32];
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) {
        const float s = attn_score(__uint_as_float(sv[jj]), i, j0 + c * 32 + jj, L, CAUSAL, bias_s, p.n_dist);
        const bool vis = i < T && s != -INFINITY;
        const float pv = vis ? ex2_approx(fmaf(s, kLog2e, -lse2)) : 0.f;
        ds[jj] = pv * (__uint_as_float(dv[jj]) - delta);
      }
      attn_store_row_chunk(smem + S::kDs, tid, c, ds);
    }
    attn_sync_for_mma();
    if (tid == 0) {
      tc_fence_after();
      attn_mma_pv(tmem, s_ds, s_k, false);  // (dS . K) of this key tile
      umma_commit<1>(&bar[1]);
    }
    attn_wait_mma(&bar[1], kt & 1);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(trow + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int d = 0; d < 32; ++d) dq[c * 32 + d] += __uint_as_float(v[d]);
    }
  }
  if (i < T) attn_store_row(p.dq + (q0 + i) * p.lddq + h * kAttnDk, dq, 1.f);  // L_b = 0: zeros
  attn_epilogue(tmem, 256, tid);
}

}  // namespace td
