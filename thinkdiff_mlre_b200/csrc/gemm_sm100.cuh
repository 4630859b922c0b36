// Persistent, warp-specialised bf16 GEMM for sm_100a: TMA -> smem ring -> tcgen05.mma (accumulators in TMEM)
// -> tcgen05.ld epilogue -> swizzled smem staging -> TMA store, with the aligner's elementwise / reduction work fused
// into the epilogue.
//
//   D[M,N] = A[M,K] * B[N,K]^T          (logical; fp32 accumulate)
//
// Each operand is either K-major (stored [rows, K], K contiguous -- activations in the forward pass, nn.Linear
// weights) or MN-major (stored [K, rows], rows contiguous -- what the backward pass has: dW = dY^T X contracts
// over the token dimension of two row-major activations, dX = dY W contracts over W's row index). The tensor
// core reads both through the 128-byte-swizzled canonical layouts, so no transposed copies are ever written.
//
// Roles (320 threads): warps 0..7 = epilogue (TMEM lane quarter = warp % 4, two warps per quarter split the columns),
// warp 8 = TMA producer, warp 9 = TMEM owner + MMA issuer. The two single-thread roles get the HIGHEST warp ids on purpose: the
// SM sub-partition schedulers favour the highest eligible warp, so the thread that feeds the tensor core is never queued behind
// the epilogue warps' GELU arithmetic on its sub-partition. CTAS=2 runs a CTA pair on one 256-row tile
// (tcgen05 cta_group::2): each CTA stages its own 128 rows of A and half of B, the leader issues the MMAs, both run their
// own epilogue.
//
// Schedule ("data-parallel waves + stream-K tail"): with W workers (CTA pairs) and T output tiles, the first
// floor(T / W) * W tiles are whole tiles, tile = wave * W + w. The remaining R = T mod W tiles would leave most workers
// idle for a whole tile time; instead their R * KB k-blocks are cut into equal contiguous ranges, one per worker. A worker
// whose range starts inside a tile is a CONTRIBUTOR for that tile: it dumps its raw fp32 accumulator to a workspace slot
// and raises a flag. The worker that holds the tile's first k-block is its OWNER: it adds the contributors' partials to
// its own accumulator in worker order (deterministic) and runs the real epilogue. No split-K memset, no atomics on the
// output, every tile is stored exactly once.
// Work is CLAIMED, not assigned: a unit is a whole tile or one tail range; every worker takes its next unit from a global
// atomic counter, so a CTA pair that becomes resident late (an SM held by a collective, an
// optimizer kernel or a flag-wait kernel of another stream) simply finds less work left instead of delaying a static share.
// Tail ranges are handed out in DESCENDING order: every contributor of a tile is claimed -- by a resident worker -- before the
// tile's owner range, so an owner never waits for work nobody is running.
//
// Reference semantics being fused (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:58-63, under the bf16
// autocast of thinkdiff/tasks/base_task.py:237): Linear -> GELU(erf) -> Linear -> T5LayerNorm, each Linear/GELU
// output rounded to bf16, the norm statistics taken in fp32 from the bf16-rounded Linear2 output.
#pragma once
#include "ptx_sm100.cuh"

namespace td {

enum EpiKind : int {
  EPI_BF16 = 0,       // out0 = bf16(acc + bias?)
  EPI_BIAS_GELU = 1,  // out0 = h0 = bf16(acc + bias) (optional); out1 = bf16(gelu(h0))
  EPI_BIAS_SSQ = 2,   // out0 = h2 = bf16(acc + bias); red0[2 * n_blk + half][row] = sum over 128 cols of h2^2
  EPI_DGELU = 3,      // t = bf16(alpha * acc); out0 = bf16(t * gelu'(aux0)); red0[m_slab * 4 + quarter][col] = sum_rows out0
  EPI_F32 = 4,        // out0(fp32) = alpha * acc
  // Row-sharded output over peer memory (data-parallel weight gradients, reduce-scatter fused into the GEMM): output row r
  // belongs to rank o = r / scatter_rows and is written to row r - o * scatter_rows of that rank's [scatter_rows, N] block -- a
  // buffer in rank o's HBM mapped into this process (the TMA bulk stores then travel over NVLink), or local memory for
  // o == this rank. One fp32 tensor map per owner; the staging and the store are those of EPI_F32.
  EPI_F32_SCATTER = 5,
  // T5 gated-GELU feed-forward (DESIGN.md section 7). The wi_0 / wi_1 rows are interleaved in blocks of 32 (t5.py), so an epilogue
  // warp's chunks 2j / 2j + 1 are a matched (a, b) pair of 32 columns: pair k = accumulator columns [64k, 64k + 64).
  EPI_GATED = 6,      // out0 = ab = bf16(acc) (optional); out1 [M, N / 2] = g = bf16(bf16(gelu_tanh(a)) * b), column 32k + i of pair k
  EPI_DGATED = 7,     // acc = dy . wo, t = bf16(acc) [M, N]; aux0 = ab [M, 2N]; out0 = d_ab [M, 2N] with, for t column 32k + i,
                      // d_a = bf16(bf16(t * b) * gelu_tanh'(a)) at column 64k + i and d_b = bf16(t * bf16(gelu_tanh(a))) at 64k + 32 + i
  EPI_RESIDUAL = 8,   // out0 = bf16(aux0 + bf16(acc)): the residual add of a sublayer's output projection
};
constexpr int kMaxPeers = 8;

struct GemmParams {
  int M, N, K;
  int num_m_blocks, num_n_blocks, num_k_blocks;  // in units of tile (BLOCK_M * CTAS, BLOCK_N, BLOCK_K)
  // schedule (filled by launch_gemm)
  int workers;       // CTA pairs (CTAS = 2) or CTAs (CTAS = 1) launched
  int full_waves;    // tiles [0, full_waves * workers) are processed whole, tile = wave * workers + worker
  int tail_workers;  // workers that share the k-blocks of the remaining tiles (0 = no tail)
  int tail_q, tail_r;  // tail worker w gets tail_q (+1 if w < tail_r) consecutive k-block units
  float* sk_partials;  // [tail ranges][CTAS][8 warps][4 chunks][32 cols][32 rows] fp32 (nullptr = tail tiles are whole tiles)
  int* sk_flags;       // [tail ranges][CTAS][8 warps] zero before the launch; re-armed by the consumer
  int* sched_counter;  // [4] zero-initialised {next unit, workers out of units, workers torn down, -}; re-armed by the kernel itself
  void* out0;
  void* out1;
  const void* aux0;
  const __nv_bfloat16* bias;
  float* red0;
  long long ld_out;  // elements
  float alpha;
  const float* alpha_ptr;  // optional device scalar multiplied into alpha (upstream loss gradient / GradScaler scale)
  float* stats;     // optional (EPI_F32 / EPI_F32_SCATTER): stats[0] += 1 per warp tile that holds a non-finite output (inf check)
  int accumulate;   // EPI_F32: out0 += alpha * acc (TMA reduce-add store; gradient accumulation over micro-batches)
  // EPI_F32_SCATTER
  float* scatter_dst[kMaxPeers];
  int scatter_rows;  // output rows per owner rank (a multiple of 32: a warp's 32-row slab never straddles two owners)
  // Raster of the output tiles (0 / 0 = groups of kGroupM m-blocks, no rotation). The scattered GEMMs of N ranks run at the same
  // time: with one common raster every rank would store to the SAME owner at the same moment (and to half of the owners for half
  // of the kernel), i.e. N senders into one NVLink port. raster_group_m = m-blocks per owner and a per-rank rotation of the
  // m-blocks turn that into a permutation: at any moment rank r stores to owner (r + 1 + t) mod N, its own rows come last.
  int raster_group_m;
  int raster_rot_m;
  // EPI_F32_SCATTER, optional: the exchange protocol's "+1 after the GEMM" folded into the GEMM itself. The last CTA pair to
  // finish (a third self-re-arming counter, sched_counter[2]) adds 1 to post_signal[o] for o < post_signal_n -- one counter in
  // every rank's memory -- after every pair's bulk stores have completed and been fenced at system scope.
  int* post_signal[kMaxPeers];
  int post_signal_n;
};
// The owners' output tensor maps of EPI_F32_SCATTER (kernel parameter; unused by the other epilogues).
struct ScatterMaps {
  CUtensorMap m[kMaxPeers];
};

constexpr int kBlockM = 128;  // rows per CTA (TMEM lanes)
constexpr int kBlockN = 256;  // accumulator columns (two stages fill the 512-column TMEM)
constexpr int kBlockK = 64;   // 64 bf16 = one 128-byte swizzle row
constexpr int kUmmaK = 16;
constexpr int kGemmThreads = 320;
#ifndef TD_ROLES_HI
#define TD_ROLES_HI 1
#endif
constexpr int kEpiWarp0 = TD_ROLES_HI ? 0 : 2;       // first of the 8 epilogue warps
constexpr int kProducerWarp = TD_ROLES_HI ? 8 : 0;   // TMA producer
constexpr int kMmaWarp = TD_ROLES_HI ? 9 : 1;        // TMEM owner + MMA issuer
constexpr int kAccStages = 2;
constexpr int kMinTailKBlocks = 8;  // a stream-K range shorter than this costs more in fix-up than it saves
// What an owner pays to fold one contributor's partial into its accumulator, in k-blocks of MMA time (plan_schedule's tail cost
// model). The fold reads 4 chunks of 4 KB per epilogue warp, one L2 round trip each, about 2 us, against about 0.3 us per k-block
// of a 256 x 256 pair tile. On a B200 (1000 W) the config-2 step measured the same with 8, 16 and 32 (dW1 0.204-0.217 ms, inside
// run-to-run noise; 0.229-0.243 ms with the old finest cut), so the estimate stands. TD_SK_FOLD_KBLOCKS overrides it for such A/Bs.
#ifndef TD_SK_FOLD_KBLOCKS
#define TD_SK_FOLD_KBLOCKS 8
#endif
constexpr int kTailFoldKBlocks = TD_SK_FOLD_KBLOCKS;

// Eight epilogue warps: warp e (0..7) owns TMEM lane quarter (warp % 4) and column half e / 4 of the 256-column
// accumulator, i.e. 32 rows x 128 columns, walked in 4 chunks of 32 columns. Thread = one output row.
constexpr int kEpiWarps = 8;
constexpr int kEpiColsPerWarp = kBlockN / (kEpiWarps / 4);  // 128
constexpr int kEpiChunks = kEpiColsPerWarp / 32;            // 4
constexpr int kSkSlotFloats = kEpiWarps * kEpiChunks * 32 * 32;  // one CTA's 128 x 256 accumulator

#ifndef TD_MAX_STAGES
#define TD_MAX_STAGES 7
#endif

// Per-warp epilogue staging in shared memory: 32-row x 32-column boxes in the layout the TMA store (or load) expects --
// 64-byte rows with the 64-byte swizzle for bf16, 128-byte rows with the 128-byte swizzle for fp32.
template <int EPI> struct EpiStage { static constexpr int kBytesPerWarp = 4096; };          // two 2 KB bf16 boxes
template <> struct EpiStage<EPI_DGELU> { static constexpr int kBytesPerWarp = 6144; };      // + two aux boxes, one out box
template <> struct EpiStage<EPI_RESIDUAL> { static constexpr int kBytesPerWarp = 6144; };   // the same layout (aux = x)
// one (d_a, d_b) output pair + two (a, b) aux pairs: 96 KB for the 8 warps leaves 4 pipeline stages
template <> struct EpiStage<EPI_DGATED> { static constexpr int kBytesPerWarp = 12288; };
// fp32 output: two 4 KB boxes, so a warp converts chunk c + 1 while the bulk store of chunk c is still reading its box -- over
// NVLink (scatter) that read is paced by the link, and a single box made the epilogue longer than the next tile's mainloop
template <> struct EpiStage<EPI_F32> { static constexpr int kBytesPerWarp = 8192; };
template <> struct EpiStage<EPI_F32_SCATTER> { static constexpr int kBytesPerWarp = 8192; };

// Pipeline depth per epilogue kind. The GEMMs that the optimizer's update kernels may run BESIDE (Linear1's update beside the dW2
// GEMM, Linear2's beside the next forward's first GEMM) keep five stages: with <= 128 registers per thread (see TD_GEMM_BOUNDS)
// and the shared memory this leaves, one 256-thread CTA of an update kernel can become resident next to the GEMM's CTA instead
// of queueing until the persistent GEMM retires. Measured (DESIGN.md section 8): where the update is full size (N = 1) running
// it beside a GEMM is no faster than running it after it -- the step is power-bound -- but in the data-parallel step it lets every
// owner finish its AdamW rows while its own dW2 GEMM still runs, so ranks that are ahead never wait for a laggard's rows.
template <int EPI> struct StageCap { static constexpr int kMax = TD_MAX_STAGES; };
#ifndef TD_NO_CORESIDENCY
template <> struct StageCap<EPI_BIAS_GELU> { static constexpr int kMax = 5; };
template <> struct StageCap<EPI_F32> { static constexpr int kMax = 5; };
template <> struct StageCap<EPI_F32_SCATTER> { static constexpr int kMax = 5; };
#endif

template <int CTAS, int EPI>
struct GemmSmem {
  static constexpr int kABytes = kBlockM * kBlockK * 2;           // 16 KB
  static constexpr int kBBytes = (kBlockN / CTAS) * kBlockK * 2;  // 32 KB or 16 KB
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kEpiBytes = kEpiWarps * EpiStage<EPI>::kBytesPerWarp;
  static constexpr int kBarrierBytes = 1024;
  static constexpr int kMaxBytes = 227 * 1024;
  static constexpr int kFit = (kMaxBytes - kBarrierBytes - 1024 - kEpiBytes) / kStageBytes;
  static constexpr int kCap = (CTAS == 2) ? StageCap<EPI>::kMax : TD_MAX_STAGES;
  static constexpr int kStages = kFit < kCap ? kFit : kCap;
  static constexpr int kTotal = kStages * kStageBytes + kEpiBytes + kBarrierBytes + 1024;  // +1024 alignment slack
  static_assert(kStages >= 3, "pipeline too shallow");
};

// ------------------------------------------------------------------------------------------ schedule
struct Segment {
  int tile;           // output tile (raster index)
  int kb0, kb1;       // k-block range of this segment
  int kind;           // 0 = whole tile / owner without contributors, 1 = owner with contributors, 2 = contributor
  int contrib0, contrib_n;  // kind 1: workers contrib0 .. contrib0 + contrib_n - 1 hold the rest of the tile
};
__host__ __device__ __forceinline__ int sk_start(const GemmParams& p, int w) { return w * p.tail_q + (w < p.tail_r ? w : p.tail_r); }
__host__ __device__ __forceinline__ int sk_worker_of(const GemmParams& p, int u) {
  const int big = p.tail_r * (p.tail_q + 1);
  return u < big ? u / (p.tail_q + 1) : p.tail_r + (u - big) / p.tail_q;
}
// Units: [0, F) = whole tiles (F = full_waves * workers, or every tile when there is no stream-K workspace), then the tail
// ranges in descending order. Calls f(segment, range) for every segment of `unit`, in execution order (a range that straddles a
// tile boundary is a contributor part followed by an owner part).
__host__ __device__ __forceinline__ int num_units(const GemmParams& p) {
  const int whole = p.tail_workers == 0 ? p.num_m_blocks * p.num_n_blocks : p.full_waves * p.workers;
  return whole + p.tail_workers;
}
template <class F>
__host__ __device__ __forceinline__ void for_each_segment(const GemmParams& p, int unit, F&& f) {
  const int KB = p.num_k_blocks;
  const int whole = p.tail_workers == 0 ? p.num_m_blocks * p.num_n_blocks : p.full_waves * p.workers;
  if (unit < whole) {
    f(Segment{unit, 0, KB, 0, 0, 0}, 0);
    return;
  }
  const int w = p.tail_workers - 1 - (unit - whole);  // tail range index
  int u = sk_start(p, w);
  const int u_end = sk_start(p, w + 1);
  while (u < u_end) {
    const int tt = u / KB;
    const int kb0 = u - tt * KB;
    const int kb1 = (kb0 + (u_end - u)) < KB ? (kb0 + (u_end - u)) : KB;
    Segment s{whole + tt, kb0, kb1, 0, 0, 0};
    if (kb0 > 0) {
      s.kind = 2;
    } else if (kb1 < KB) {
      s.kind = 1;
      s.contrib0 = w + 1;
      s.contrib_n = sk_worker_of(p, (tt + 1) * KB - 1) - w;
    }
    f(s, w);
    u += kb1 - kb0;
  }
}

constexpr int kGroupM = 8;  // rasterise m-blocks in groups so that concurrently running tiles share operands in L2
__host__ __device__ __forceinline__ void tile_coords(const GemmParams& p, int tile, int& m_blk, int& n_blk) {
  const int nnb = p.num_n_blocks;
  const int G = p.raster_group_m > 0 ? p.raster_group_m : kGroupM;
  const int group = tile / (G * nnb);
  const int first_m = group * G;
  const int rest_m = p.num_m_blocks - first_m;
  const int gsize = G < rest_m ? G : rest_m;
  const int in_group = tile - group * G * nnb;
  m_blk = first_m + in_group % gsize;
  n_blk = in_group / gsize;
  if (p.raster_rot_m > 0) {
    m_blk += p.raster_rot_m;
    if (m_blk >= p.num_m_blocks) m_blk -= p.num_m_blocks;
  }
}

// ------------------------------------------------------------------------------------------ epilogue helpers
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  f[0] = bf16lo(u.x); f[1] = bf16hi(u.x); f[2] = bf16lo(u.y); f[3] = bf16hi(u.y);
  f[4] = bf16lo(u.z); f[5] = bf16hi(u.z); f[6] = bf16lo(u.w); f[7] = bf16hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}
// Byte offset of 16-byte piece q of row r inside a 32-row staging box.
__device__ __forceinline__ uint32_t box64_off(int r, int q) {   // 64-byte rows, CU_TENSOR_MAP_SWIZZLE_64B
  return uint32_t(r * 64 + ((q ^ ((r >> 1) & 3)) << 4));
}
__device__ __forceinline__ uint32_t box128_off(int r, int q) {  // 128-byte rows, CU_TENSOR_MAP_SWIZZLE_128B
  return uint32_t(r * 128 + ((q ^ (r & 7)) << 4));
}

// State an epilogue warp carries from tile to tile.
struct EpiState {
  uint32_t box;      // staging boxes written so far (parity selects the buffer)
  uint32_t aux_req;  // aux boxes requested so far (EPI_DGELU); box n lands in buffer n & 1, barrier parity (n >> 1) & 1
  uint32_t aux_use;  // aux boxes consumed so far
};

// Hand a filled staging box to the TMA: make the generic-proxy writes visible to the async proxy, then one lane stores.
__device__ __forceinline__ void stage_store(const CUtensorMap* map, const void* box, int col0, int row0, int lane,
                                            bool reduce_add = false) {
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    if (reduce_add) tma_reduce_add_2d(map, box, col0, row0); else tma_store_2d(map, box, col0, row0);
    tma_store_commit();
  }
}
// Before a staging box is overwritten: the bulk store issued two boxes ago (same buffer) must have read it.
__device__ __forceinline__ void stage_acquire(int lane, bool single_buffer) {
  if (lane == 0) {
    if (single_buffer) tma_store_wait_read<0>(); else tma_store_wait_read<1>();
  }
  __syncwarp();
}

template <int CTAS, int EPI>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, const CUtensorMap* map_out0, const CUtensorMap* map_out1,
                                              const CUtensorMap* map_aux, const ScatterMaps& smaps, uint8_t* stage, uint64_t* aux_bar,
                                              EpiState& st,
                                              const Segment& seg, uint32_t tmem_acc, int row0, int n0, int n_blk, int m_slab,
                                              int quarter, int half, int lane, int range, uint32_t cta_rank, int e) {
  const int row = row0 + quarter * 32 + lane;
  const bool row_ok = row < p.M;
  const int slab_row0 = row0 + quarter * 32;
  const int ncol0 = n0 + half * kEpiColsPerWarp;
  const uint32_t taddr = tmem_acc + (uint32_t(quarter * 32) << 16) + half * kEpiColsPerWarp;

  // ---- contributor: dump the raw accumulator, coalesced (lane = consecutive floats), and raise this warp's flag
  if (seg.kind == 2) {
    float* slot = p.sk_partials + ((size_t)(range * CTAS + cta_rank) * kEpiWarps + e) * (kEpiChunks * 1024);
#pragma unroll 1
    for (int c = 0; c < kEpiChunks; ++c) {
      if (ncol0 + c * 32 >= p.N) break;
      uint32_t v[32];
      tmem_ld_32x32(taddr + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) slot[c * 1024 + j * 32 + lane] = __uint_as_float(v[j]);
    }
    __threadfence();
    __syncwarp();
    if (lane == 0) st_release_gpu(p.sk_flags + (range * CTAS + cta_rank) * kEpiWarps + e, 1);
    return;
  }
  // ---- owner of a shared tile: wait until every contributor's warp `e` has published its partial
  if (seg.kind == 1) {
    if (lane == 0) {
      for (int i = 0; i < seg.contrib_n; ++i)
        spin_until_set(p.sk_flags + ((seg.contrib0 + i) * CTAS + cta_rank) * kEpiWarps + e);
    }
    __syncwarp();
  }

  float ssq = 0.f;
  bool bad = false;  // EPI_F32 / EPI_F32_SCATTER: a non-finite output was produced (GradScaler's inf check)
  float alpha = p.alpha;
  if constexpr (EPI == EPI_F32 || EPI == EPI_DGELU || EPI == EPI_F32_SCATTER) {
    if (p.alpha_ptr != nullptr) alpha *= __ldg(p.alpha_ptr);
  }

  // EPI_DGELU: the saved pre-activation h0 arrives by TMA, one 32 x 32 box per chunk, one box ahead of the math (EPI_RESIDUAL: x).
  // EPI_DGATED: the (a, b) box pair of chunk c, columns 2 col0 and 2 col0 + 32 of ab, at +4096 / +8192; the output pair is at +0.
  constexpr bool kAux = EPI == EPI_DGELU || EPI == EPI_RESIDUAL || EPI == EPI_DGATED;
  uint8_t* aux_box = stage + (EPI == EPI_DGATED ? 4096 : 2048);  // otherwise boxes at +2048 and +4096; the output box is at +0
  auto aux_request = [&](int c) {
    if (lane == 0) {
      const uint32_t b = st.aux_req & 1;
      if constexpr (EPI == EPI_DGATED) {
        const int ab_col = 2 * (ncol0 + c * 32);
        mbar_arrive_expect_tx(&aux_bar[b], 4096);
        tma_load_2d(aux_box + b * 4096, map_aux, &aux_bar[b], ab_col, slab_row0);
        tma_load_2d(aux_box + b * 4096 + 2048, map_aux, &aux_bar[b], ab_col + 32, slab_row0);
      } else {
        mbar_arrive_expect_tx(&aux_bar[b], 2048);
        tma_load_2d(aux_box + b * 2048, map_aux, &aux_bar[b], ncol0 + c * 32, slab_row0);
      }
    }
    st.aux_req++;
  };
  if constexpr (kAux) {
    if (ncol0 < p.N) aux_request(0);
  }
  float gate[EPI == EPI_GATED ? 32 : 1];  // EPI_GATED: bf16(gelu_tanh(a)) of the last a chunk, for the b chunk that follows it

#pragma unroll 1
  for (int c = 0; c < kEpiChunks; ++c) {
    const int col0 = ncol0 + c * 32;
    if (col0 >= p.N) break;  // N % 32 == 0 is enforced on the host
    uint32_t v[32];
    tmem_ld_32x32(taddr + c * 32, v);
    if constexpr (kAux) {
      if (c + 1 < kEpiChunks && col0 + 32 < p.N) aux_request(c + 1);
    }
    tmem_ld_wait();
    if (seg.kind == 1) {
      for (int i = 0; i < seg.contrib_n; ++i) {
        const float* part = p.sk_partials + ((size_t)((seg.contrib0 + i) * CTAS + cta_rank) * kEpiWarps + e) * (kEpiChunks * 1024) + c * 1024;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __ldcg(part + j * 32 + lane));
      }
    }

    if constexpr (EPI == EPI_F32_SCATTER || EPI == EPI_F32) {
      const CUtensorMap* map = map_out0;
      int out_row0 = slab_row0;
      if constexpr (EPI == EPI_F32_SCATTER) {
        if (slab_row0 >= p.M) continue;                // rows past M belong to no owner (the plain store is clipped by its map)
        const int owner = slab_row0 / p.scatter_rows;  // warp-uniform
        map = &smaps.m[owner];
        out_row0 = slab_row0 - owner * p.scatter_rows;
      }
      uint8_t* box = stage + (st.box & 1) * 4096;
      stage_acquire(lane, false);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          o[j] = alpha * __uint_as_float(v[4 * q + j]);
          bad |= row_ok && !(fabsf(o[j]) <= 3.4028234e38f);
        }
        *reinterpret_cast<uint4*>(box + box128_off(lane, q)) =
            make_uint4(__float_as_uint(o[0]), __float_as_uint(o[1]), __float_as_uint(o[2]), __float_as_uint(o[3]));
      }
      stage_store(map, box, col0, out_row0, lane, EPI == EPI_F32 && p.accumulate != 0);
      st.box++;
    } else if constexpr (EPI == EPI_DGELU) {
      // dh0 = bf16( bf16(dh1) * gelu'(h0) ): dh1 is rounded to bf16 first, as autograd materialises it.
      const uint32_t b = st.aux_use & 1;
      mbar_wait(&aux_bar[b], (st.aux_use >> 1) & 1);
      st.aux_use++;
      // Rows past M need no predicate: their A rows and their aux box are zero-filled by the TMA, so t = 0 and the output is
      // 0 * gelu'(0) = 0. Rounding to bf16 goes through the packed conversion (two values per ALU-pipe instruction).
      float colsum[32];
      uint4 outp[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float x[8];
        uint32_t w[4];
        unpack8(*reinterpret_cast<const uint4*>(aux_box + b * 2048 + box64_off(lane, q)), x);
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          float t0 = alpha * __uint_as_float(v[q * 8 + j]), t1 = alpha * __uint_as_float(v[q * 8 + j + 1]);
          bf16_round2(t0, t1);
          float h0 = t0 * gelu_grad_fast(x[j]), h1 = t1 * gelu_grad_fast(x[j + 1]);
          w[j >> 1] = bf16_round2(h0, h1);
          colsum[q * 8 + j] = h0;
          colsum[q * 8 + j + 1] = h1;
        }
        outp[q] = make_uint4(w[0], w[1], w[2], w[3]);
      }
      stage_acquire(lane, true);  // (also orders every lane's aux reads before the next request overwrites that box)
#pragma unroll
      for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(stage + box64_off(lane, q)) = outp[q];
      stage_store(map_out0, stage, col0, slab_row0, lane);
      // Column sums over this warp's 32 rows by a butterfly transpose-reduce: after the 5 rounds lane j holds
      // the sum over lanes of colsum[j]. 31 shuffles for 32 columns.
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
          const float send = upper ? colsum[i] : colsum[i + off];
          const float keep = upper ? colsum[i + off] : colsum[i];
          colsum[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      p.red0[(long long)(m_slab * 4 + quarter) * p.N + col0 + lane] = colsum[0];
    } else if constexpr (EPI == EPI_RESIDUAL) {
      const uint32_t b = st.aux_use & 1;
      mbar_wait(&aux_bar[b], (st.aux_use >> 1) & 1);
      st.aux_use++;
      uint4 outp[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float x[8];
        uint32_t w[4];
        unpack8(*reinterpret_cast<const uint4*>(aux_box + b * 2048 + box64_off(lane, q)), x);
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          float f0 = __uint_as_float(v[q * 8 + j]), f1 = __uint_as_float(v[q * 8 + j + 1]);
          bf16_round2(f0, f1);  // the projection's output is a bf16 tensor before the add
          w[j >> 1] = pack_bf16x2(x[j] + f0, x[j + 1] + f1);
        }
        outp[q] = make_uint4(w[0], w[1], w[2], w[3]);
      }
      stage_acquire(lane, true);  // (also orders every lane's aux reads before the next request overwrites that box)
#pragma unroll
      for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(stage + box64_off(lane, q)) = outp[q];
      stage_store(map_out0, stage, col0, slab_row0, lane);
    } else if constexpr (EPI == EPI_DGATED) {
      // Rows past M: their A rows and aux boxes are zero-filled, so every output is 0 (and the store clips them anyway).
      const uint32_t b = st.aux_use & 1;
      mbar_wait(&aux_bar[b], (st.aux_use >> 1) & 1);
      st.aux_use++;
      const uint8_t* a_box = aux_box + b * 4096;
      uint4 out_a[4], out_b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float av[8], bv[8];
        uint32_t wa[4], wb[4];
        unpack8(*reinterpret_cast<const uint4*>(a_box + box64_off(lane, q)), av);
        unpack8(*reinterpret_cast<const uint4*>(a_box + 2048 + box64_off(lane, q)), bv);
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          float t0 = __uint_as_float(v[q * 8 + j]), t1 = __uint_as_float(v[q * 8 + j + 1]);
          bf16_round2(t0, t1);  // t = dL/dg, a bf16 tensor in autograd
          float g0, g1;
          const float d0 = gelu_tanh_grad(av[j], g0), d1 = gelu_tanh_grad(av[j + 1], g1);
          bf16_round2(g0, g1);  // gelu(a) as the forward materialised it
          wb[j >> 1] = pack_bf16x2(t0 * g0, t1 * g1);
          float u0 = t0 * bv[j], u1 = t1 * bv[j + 1];
          bf16_round2(u0, u1);  // dL/dgelu(a)
          wa[j >> 1] = pack_bf16x2(u0 * d0, u1 * d1);
        }
        out_a[q] = make_uint4(wa[0], wa[1], wa[2], wa[3]);
        out_b[q] = make_uint4(wb[0], wb[1], wb[2], wb[3]);
      }
      stage_acquire(lane, true);  // the previous pair's stores have read their boxes; orders the aux reads as above
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        *reinterpret_cast<uint4*>(stage + box64_off(lane, q)) = out_a[q];
        *reinterpret_cast<uint4*>(stage + 2048 + box64_off(lane, q)) = out_b[q];
      }
      stage_store(map_out0, stage, 2 * col0, slab_row0, lane);
      stage_store(map_out0, stage + 2048, 2 * col0 + 32, slab_row0, lane);
    } else if constexpr (EPI == EPI_GATED) {
      // chunk c even: a (wi_0 rows), keep bf16(gelu_tanh(a)); c odd: the matching b (wi_1 rows), emit g. N % 64 == 0 and
      // ncol0 % 64 == 0, so an a chunk inside N is always followed by its b chunk.
      const bool is_b = (c & 1) != 0;
      uint4 o0[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t w0[4];
#pragma unroll
        for (int j = 0; j < 8; j += 2) w0[j >> 1] = pack_bf16x2(__uint_as_float(v[q * 8 + j]), __uint_as_float(v[q * 8 + j + 1]));
        o0[q] = make_uint4(w0[0], w0[1], w0[2], w0[3]);
      }
      if (!is_b) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float a[8];
          unpack8(o0[q], a);
#pragma unroll
          for (int j = 0; j < 8; j += 2) {
            float g0 = gelu_tanh(a[j]), g1 = gelu_tanh(a[j + 1]);
            bf16_round2(g0, g1);
            gate[q * 8 + j] = g0;
            gate[q * 8 + j + 1] = g1;
          }
        }
      }
      if (p.out0 != nullptr) {  // inference skips saving a and b
        uint8_t* box = stage + (st.box & 1) * 2048;
        stage_acquire(lane, false);
#pragma unroll
        for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(box + box64_off(lane, q)) = o0[q];
        stage_store(map_out0, box, col0, slab_row0, lane);
        st.box++;
      }
      if (is_b) {
        uint4 o1[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float b[8];
          uint32_t w1[4];
          unpack8(o0[q], b);
#pragma unroll
          for (int j = 0; j < 8; j += 2) w1[j >> 1] = pack_bf16x2(gate[q * 8 + j] * b[j], gate[q * 8 + j + 1] * b[j + 1]);
          o1[q] = make_uint4(w1[0], w1[1], w1[2], w1[3]);
        }
        uint8_t* box = stage + (st.box & 1) * 2048;
        stage_acquire(lane, false);
#pragma unroll
        for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(box + box64_off(lane, q)) = o1[q];
        stage_store(map_out1, box, (col0 - 32) >> 1, slab_row0, lane);
        st.box++;
      }
    } else {
      // bias (bf16, same 32 columns for every thread of the warp -> broadcast loads)
      uint4 o0[4], o1[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float b[8], h[8];
        uint32_t w0[4], w1[4];
        if (p.bias != nullptr) {
          unpack8(__ldg(reinterpret_cast<const uint4*>(p.bias + col0) + q), b);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) b[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; j += 2) {  // bf16 rounding through the packed conversion (ALU pipe), two values at a time
          h[j] = __uint_as_float(v[q * 8 + j]) + b[j];
          h[j + 1] = __uint_as_float(v[q * 8 + j + 1]) + b[j + 1];
          w0[j >> 1] = bf16_round2(h[j], h[j + 1]);
        }
        o0[q] = make_uint4(w0[0], w0[1], w0[2], w0[3]);
        if constexpr (EPI == EPI_BIAS_GELU) {
#pragma unroll
          for (int j = 0; j < 8; j += 2) w1[j >> 1] = pack_bf16x2(gelu_fast(h[j]), gelu_fast(h[j + 1]));
          o1[q] = make_uint4(w1[0], w1[1], w1[2], w1[3]);
        }
        if constexpr (EPI == EPI_BIAS_SSQ) {
#pragma unroll
          for (int j = 0; j < 8; ++j) ssq = fmaf(h[j], h[j], ssq);
        }
      }
      if (p.out0 != nullptr) {  // inference skips saving the pre-activation
        uint8_t* box = stage + (st.box & 1) * 2048;
        stage_acquire(lane, false);
#pragma unroll
        for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(box + box64_off(lane, q)) = o0[q];
        stage_store(map_out0, box, col0, slab_row0, lane);
        st.box++;
      }
      if constexpr (EPI == EPI_BIAS_GELU) {
        uint8_t* box = stage + (st.box & 1) * 2048;
        stage_acquire(lane, false);
#pragma unroll
        for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(box + box64_off(lane, q)) = o1[q];
        stage_store(map_out1, box, col0, slab_row0, lane);
        st.box++;
      }
    }
  }
  if constexpr (EPI == EPI_BIAS_SSQ) {
    if (row_ok) p.red0[(long long)(n_blk * 2 + half) * p.M + row] = ssq;
  }
  if constexpr (EPI == EPI_F32 || EPI == EPI_F32_SCATTER) {
    if (p.stats != nullptr && __any_sync(0xffffffffu, bad) && lane == 0) atomicAdd(p.stats, 1.0f);
  }
  if (seg.kind == 1) {  // re-arm the flags this warp consumed: the pool slot is zero again for a later launch
    __syncwarp();
    if (lane == 0) {
      for (int i = 0; i < seg.contrib_n; ++i) p.sk_flags[((seg.contrib0 + i) * CTAS + cta_rank) * kEpiWarps + e] = 0;
    }
  }
}

// ------------------------------------------------------------------------------------------ kernel
// Work distribution: the leader's producer thread claims units from a global atomic counter (the claim for the NEXT unit is
// issued before the current unit's loads, hiding the atomic's round trip) and publishes each claim through a small shared-memory ring (`sched_*`) to the MMA thread and the epilogue warps
// -- and, for a pair, to the peer CTA over DSMEM.
constexpr int kSchedStages = 4;

// Register budget. A warp's registers come from its SM sub-partition's quarter of the register file (16 384 x 32 bit): the ten
// GEMM warps put three on sub-partitions 0 and 1, so at more than 128 registers per thread (allocated in units of 8) there is no
// room left there for even two warps of a co-resident 256-thread update kernel at 64 registers (3 x 32 x 128 + 2 x 32 x 64 =
// 16 384 exactly) -- it then sits in the block scheduler until the GEMM's CTAs exit. The fp32-output epilogues compile to
// 124-126 registers; TD_GEMM_MAXNREG caps every instantiation (developer A/B: with it the N = 1 step was 2.5 % SLOWER).
#ifdef TD_GEMM_MAXNREG
#define TD_GEMM_BOUNDS __maxnreg__(TD_GEMM_MAXNREG)
#else
#define TD_GEMM_BOUNDS __launch_bounds__(kGemmThreads, 1)
#endif
template <int CTAS, bool A_MN, bool B_MN, int EPI>
__global__ void TD_GEMM_BOUNDS
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_out0, const __grid_constant__ CUtensorMap tmap_out1,
                 const __grid_constant__ CUtensorMap tmap_aux, const __grid_constant__ ScatterMaps smaps, const GemmParams p) {
  using S = GemmSmem<CTAS, EPI>;
  constexpr int kStages = S::kStages;
  constexpr int kBRows = kBlockN / CTAS;  // B rows staged by one CTA

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* epi_smem = smem + kStages * S::kStageBytes;  // 1024-byte aligned (stage sizes are multiples of 16 KB)
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem + S::kEpiBytes);
  uint64_t* full_bar = bars;                                  // [kStages]   TMA -> MMA
  uint64_t* empty_bar = full_bar + kStages;                   // [kStages]   MMA -> TMA
  uint64_t* acc_full_bar = empty_bar + kStages;               // [kAccStages] MMA -> epilogue
  uint64_t* acc_empty_bar = acc_full_bar + kAccStages;        // [kAccStages] epilogue -> MMA
  uint64_t* aux_bar = acc_empty_bar + kAccStages;             // [kEpiWarps][2] TMA (aux boxes) -> epilogue warp
  uint64_t* sched_full_bar = aux_bar + 2 * kEpiWarps;         // [kSchedStages] scheduler -> consumers
  uint64_t* sched_empty_bar = sched_full_bar + kSchedStages;  // [kSchedStages] consumers -> scheduler (leader's copy is used)
  int* sched_unit = reinterpret_cast<int*>(sched_empty_bar + kSchedStages);  // [kSchedStages]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sched_unit + kSchedStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CTAS == 2) ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  // consumers of a published unit, per CTA: 8 epilogue warps + 1 (the MMA thread in the leader, the producer in the peer)
  constexpr uint32_t kSchedConsumers = (kEpiWarps + 1) * CTAS;

  if (warp == kProducerWarp && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if constexpr (EPI != EPI_F32_SCATTER) tma_prefetch_desc(&tmap_out0);
    else tma_prefetch_desc(&smaps.m[0]);
    if constexpr (EPI == EPI_BIAS_GELU || EPI == EPI_GATED) tma_prefetch_desc(&tmap_out1);
    if constexpr (EPI == EPI_DGELU || EPI == EPI_RESIDUAL || EPI == EPI_DGATED) tma_prefetch_desc(&tmap_aux);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(&acc_full_bar[s], 1);
      mbar_init(&acc_empty_bar[s], kEpiWarps * CTAS);
    }
    for (int s = 0; s < 2 * kEpiWarps; ++s) mbar_init(&aux_bar[s], 1);
    for (int s = 0; s < kSchedStages; ++s) {
      mbar_init(&sched_full_bar[s], 1);
      mbar_init(&sched_empty_bar[s], kSchedConsumers);
    }
    fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc<CTAS>(tmem_slot, 512);
    tmem_relinquish<CTAS>();
  }
  tc_fence_before();
  if constexpr (CTAS == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  // Everything above touches only this CTA's (or pair's) shared memory, TMEM and kernel parameters, so it may run under the
  // previous kernel's tail (programmatic dependent launch). The scheduler counter, every TMA load, the bias / alpha_ptr /
  // stream-K flag reads and every store come after the wait.
  grid_dependency_wait();
  const uint32_t tmem_base = *tmem_slot;
  const int num_workers = gridDim.x / CTAS;
  const int n_units = num_units(p);

  // consumer side of the scheduler ring: wait for slot `ss`, read the unit, release the slot (one arrive per warp)
  auto sched_consume = [&](int ss, uint32_t sphase, bool whole_warp) -> int {
    mbar_wait_cluster(&sched_full_bar[ss], sphase);
    const int unit = *reinterpret_cast<volatile int*>(&sched_unit[ss]);
    if (whole_warp) __syncwarp();
    if (!whole_warp || lane == 0) {
      if constexpr (CTAS == 1) mbar_arrive(&sched_empty_bar[ss]);
      else mbar_arrive_cluster(&sched_empty_bar[ss], 0);
    }
    return unit;
  };

  if (warp == kProducerWarp) {
    // ===================================================== scheduler + TMA producer
    if (lane == 0) {
      int stage = 0, ss = 0;
      uint32_t phase = 0, sphase = 0;
      // EVERY unit is claimed, the first one too: only a worker that is actually running can hold a unit, which is what makes
      // the stream-K owner/contributor waits deadlock-free when some CTA pairs cannot become resident for a while
      int claimed = leader ? atomicAdd(p.sched_counter, 1) : 0;
      while (true) {
        int unit;
        if (leader) {
          unit = claimed;
          if (unit < n_units) claimed = atomicAdd(p.sched_counter, 1);
          if (unit >= n_units) unit = -1;
          mbar_wait_cluster(&sched_empty_bar[ss], sphase ^ 1);  // every consumer (both CTAs) has read the old value
          sched_unit[ss] = unit;
          mbar_arrive(&sched_full_bar[ss]);  // release.cta: orders the store above for this CTA's consumers
          if constexpr (CTAS == 2) {
            st_shared_cluster_s32(&sched_unit[ss], 1, unit);
            mbar_arrive_cluster(&sched_full_bar[ss], 1);  // release.cluster: orders the remote store
          }
        } else {
          unit = sched_consume(ss, sphase, false);
        }
        if (++ss == kSchedStages) { ss = 0; sphase ^= 1; }
        if (unit < 0) break;
        for_each_segment(p, unit, [&](const Segment& seg, int) {
          int m_blk, n_blk;
          tile_coords(p, seg.tile, m_blk, n_blk);
          const int a_row0 = m_blk * (kBlockM * CTAS) + cta_rank * kBlockM;
          const int b_row0 = n_blk * kBlockN + cta_rank * kBRows;
          for (int kb = seg.kb0; kb < seg.kb1; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * S::kStageBytes;
            uint8_t* sb = sa + S::kABytes;
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], S::kStageBytes * CTAS);
            const int k0 = kb * kBlockK;
            if constexpr (!A_MN) {
              if constexpr (CTAS == 1) tma_load_2d(sa, &tmap_a, &full_bar[stage], k0, a_row0);
              else tma_load_2d_pair(sa, &tmap_a, &full_bar[stage], k0, a_row0);
            } else {
#pragma unroll
              for (int j = 0; j < kBlockM / 64; ++j) {
                if constexpr (CTAS == 1) tma_load_2d(sa + j * (kBlockK * 128), &tmap_a, &full_bar[stage], a_row0 + j * 64, k0);
                else tma_load_2d_pair(sa + j * (kBlockK * 128), &tmap_a, &full_bar[stage], a_row0 + j * 64, k0);
              }
            }
            if constexpr (!B_MN) {
              if constexpr (CTAS == 1) tma_load_2d(sb, &tmap_b, &full_bar[stage], k0, b_row0);
              else tma_load_2d_pair(sb, &tmap_b, &full_bar[stage], k0, b_row0);
            } else {
#pragma unroll
              for (int j = 0; j < kBRows / 64; ++j) {
                if constexpr (CTAS == 1) tma_load_2d(sb + j * (kBlockK * 128), &tmap_b, &full_bar[stage], b_row0 + j * 64, k0);
                else tma_load_2d_pair(sb + j * (kBlockK * 128), &tmap_b, &full_bar[stage], b_row0 + j * 64, k0);
              }
            }
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        });
      }
      // this worker has no unit left: the next kernel of the stream may start its prologue on the SMs that free up
      grid_launch_dependents();
      if (leader) {
        // the last worker to run out of units re-arms the counter pair for the next launch that uses this slot
        __threadfence();
        if (atomicAdd(p.sched_counter + 1, 1) == num_workers - 1) {
          p.sched_counter[0] = 0;
          p.sched_counter[1] = 0;
          __threadfence();
        }
      }
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // ===================================================== MMA issuer (leader CTA only)
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(kBlockM * CTAS, kBlockN, A_MN, B_MN);
      // K-major SW128: rows 128 B apart, 8-row groups 1024 B apart (SBO); LBO unused.
      // MN-major SW128: 64-element row chunks; next 8 k-rows 1024 B (SBO), next 64 MN elements one box (LBO).
      constexpr uint32_t a_lbo = A_MN ? kBlockK * 128 : 16, b_lbo = B_MN ? kBlockK * 128 : 16;
      constexpr uint32_t sbo = 1024;
      constexpr uint32_t a_kstep = A_MN ? kUmmaK * 128 : kUmmaK * 2;  // bytes per UMMA_K step
      constexpr uint32_t b_kstep = B_MN ? kUmmaK * 128 : kUmmaK * 2;
      int stage = 0, acc = 0, ss = 0;
      uint32_t phase = 0, acc_phase = 0, sphase = 0;
      while (true) {
        const int unit = sched_consume(ss, sphase, false);
        if (++ss == kSchedStages) { ss = 0; sphase ^= 1; }
        if (unit < 0) break;
        for_each_segment(p, unit, [&](const Segment& seg, int) {
          mbar_wait(&acc_empty_bar[acc], acc_phase ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + acc * kBlockN;
          for (int kb = seg.kb0; kb < seg.kb1; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + stage * S::kStageBytes);
            const uint32_t sb = sa + S::kABytes;
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              const uint64_t adesc = make_smem_desc_sw128(sa + k * a_kstep, a_lbo, sbo);
              const uint64_t bdesc = make_smem_desc_sw128(sb + k * b_kstep, b_lbo, sbo);
              umma_bf16<CTAS>(tmem_d, adesc, bdesc, idesc, (kb > seg.kb0 || k > 0) ? 1u : 0u);
            }
            umma_commit<CTAS>(&empty_bar[stage]);  // smem slot reusable once these MMAs have read it
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
          umma_commit<CTAS>(&acc_full_bar[acc]);  // accumulator complete -> epilogue(s)
          if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
        });
      }
    }
    __syncwarp();
  } else {
    // ===================================================== epilogue warps (TMEM lane quarter = warp % 4)
    const int quarter = warp & 3;
    const int e = warp - kEpiWarp0;
    const int half = e >> 2;
    uint8_t* stage = epi_smem + e * EpiStage<EPI>::kBytesPerWarp;
    EpiState st{0u, 0u, 0u};
    int acc = 0, ss = 0;
    uint32_t acc_phase = 0, sphase = 0;
    while (true) {
      const int unit = sched_consume(ss, sphase, true);
      if (++ss == kSchedStages) { ss = 0; sphase ^= 1; }
      if (unit < 0) break;
      for_each_segment(p, unit, [&](const Segment& seg, int range) {
        int m_blk, n_blk;
        tile_coords(p, seg.tile, m_blk, n_blk);
        mbar_wait(&acc_full_bar[acc], acc_phase);
        tc_fence_after();
        const int m_slab = m_blk * CTAS + cta_rank;
        epilogue_tile<CTAS, EPI>(p, &tmap_out0, &tmap_out1, &tmap_aux, smaps, stage, aux_bar + 2 * e, st, seg, tmem_base + acc * kBlockN,
                                 m_slab * kBlockM, n_blk * kBlockN, n_blk, m_slab, quarter, half, lane, range, cta_rank, e);
        tc_fence_before();
        __syncwarp();  // all 32 lanes have drained their TMEM loads; one (release) arrive per warp
        if (lane == 0) {
          if constexpr (CTAS == 1) mbar_arrive(&acc_empty_bar[acc]);
          else mbar_arrive_cluster(&acc_empty_bar[acc], 0);
        }
        if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
      });
    }
    if (lane == 0) {
      tma_store_wait_all<0>();  // the staging boxes must outlive the bulk stores that read them
      if constexpr (EPI == EPI_F32_SCATTER) __threadfence_system();  // peer-memory stores: complete before the kernel is
    }
  }

  // teardown: everyone (both CTAs of a pair) must be done with TMEM and the barriers before it is freed
  tc_fence_before();
  if constexpr (CTAS == 2) cluster_sync_all(); else __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc<CTAS>(tmem_base, 512);
  }
  if constexpr (EPI == EPI_F32_SCATTER) {
    // Every epilogue warp of this pair has waited for its bulk stores and fenced at system scope before the barrier above. The
    // worker that finds all others already here publishes the whole GEMM: release at system scope, one counter per rank.
    if (p.post_signal_n > 0 && leader && warp == kProducerWarp && lane == 0) {
      __threadfence();
      if (atomicAdd(p.sched_counter + 2, 1) == num_workers - 1) {
        p.sched_counter[2] = 0;
        __threadfence_system();
#pragma unroll
        for (int o = 0; o < kMaxPeers; ++o)
          if (o < p.post_signal_n) asm volatile("red.release.sys.global.add.s32 [%0], 1;" ::"l"(p.post_signal[o]) : "memory");
      }
    }
  }
}

}  // namespace td
