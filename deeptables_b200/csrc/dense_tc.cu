// Dense-layer GEMMs on the 5th-generation tensor cores (tcgen05 + TMEM): keras Dense forward / data gradient /
// weight gradient (dnn() tower, deepnets.py:401-427; per-net logit layers wider than 8, deepmodel.py:292; the AutoInt
// Q/K/V/residual projections, layers.py:106-127) and the GEMMs of the any-shape CIN formulation (cin_fp32.cu).
//
// fp32 in, fp32 out.  Operands are split on the fly into bf16 hi + lo and multiplied in three tensor passes
// (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM): each operand is represented to 2^-18, the dropped lo*lo term is
// 2^-18 of a product, i.e. fp32-grade results (the same scheme the CIN kernels use, cin_tc.cu).
//
//   rows kernel   out[M, Nout] = act(A[M, K] . W + bias)       W given as packed images (dense_tc_pack_kernel)
//                 forward:   A = X,  W = kernel          [K = in_dim,  Nout = out_dim]
//                 dgrad:     A = dZ, W = kernel^T        [K = out_dim, Nout = in_dim]
//   wgrad kernel  dW[K, N] += sum_m X[m, k] dZ[m, n]     both operands converted on the fly; reduction over batch rows
//
// These shapes are HBM-bound (126 kFLOP per 1.7 KB row for 429 -> 128 -> 64), so the structure is a streaming one:
// coalesced fp32 reads -> registers -> bf16 hi/lo core matrices in shared memory (UMMA canonical K-major, no swizzle)
// -> tcgen05.mma (SS form), 4-stage mbarrier ring, weights by bulk async copy, double-buffered TMEM accumulators whose
// read-out (bias / relu; lane = output row, 32 columns per TMEM read written as 8 float4 of the lane's own 128-byte line)
// overlaps the next tile's loads.  Outputs whose rows are not 16-byte aligned go through a shared-memory transpose instead
// (it was the only form until the [B*F, 32] -> 128 AutoInt projection measured 0.82 ms against 0.44 ms for the direct
// stores).
#include "dtb_common.cuh"
#include "tcgen05.cuh"
#include "dense_tc.h"
#include <cuda_bf16.h>

namespace dtb {

constexpr int kDtThreads = 448;        // rows kernel: warps 0-7 producers, 8-11 epilogue, 12 MMA issue + TMEM owner, 13 weight loader
constexpr int kDtWgThreads = 320;      // wgrad kernel: warps 0-3 X producers (+ epilogue), 4-7 dZ producers, 8 MMA issue
constexpr int kDtKc = 32;              // reduction elements per pipeline stage (two UMMA k-steps)
constexpr int kDtStages = 4;
constexpr int kDtAImg = 128 * kDtKc * 2;          // bytes of one bf16 [128 x 32] image
constexpr int kDtAStage = 2 * kDtAImg;            // hi + lo
constexpr int kDtMaxNT = 256;

static inline int dt_round_up(int x, int m) { return (x + m - 1) / m * m; }

// ------------------------------------------------------------------------------------------
// weight pack: fp32 W (row-major, leading dimension ldw) -> per (n-tile, k-chunk) [hi image | lo image],
// image = canonical K-major no-swizzle tile of B[n][kk]:  core (kk/8, n/8) at ((kk/8)*(NT/8) + n/8)*128 B,
// row n%8 at 16 B, element kk%8 at 2 B.   transposed = 0: B[n][kk] = W[(k0+kk)*ldw + n0+n]   (forward)
//                                         transposed = 1: B[n][kk] = W[(n0+n)*ldw + k0+kk]   (data gradient)
// ------------------------------------------------------------------------------------------
__global__ void dense_tc_pack_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int K, int N, int ldw,
                                     int NT, int n_tiles, int n_chunks, int transposed) {
  const int64_t per_chunk = (int64_t)NT * kDtKc;
  const int64_t total = per_chunk * n_chunks * n_tiles;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t img = t / per_chunk;
    const int rem = (int)(t - img * per_chunk);
    const int nt = (int)(img / n_chunks), c = (int)(img - (int64_t)nt * n_chunks);
    int kk, n;
    if (transposed) { n = rem / kDtKc; kk = rem - n * kDtKc; }     // kk fastest: coalesced reads of W rows
    else            { kk = rem / NT;   n = rem - kk * NT; }        // n fastest
    const int k = c * kDtKc + kk, col = nt * NT + n;
    float v = 0.f;
    if (k < K && col < N) v = transposed ? w[(int64_t)col * ldw + k] : w[(int64_t)k * ldw + col];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    const int64_t off = ((int64_t)(kk >> 3) * (NT >> 3) + (n >> 3)) * 128 + (n & 7) * 16 + (kk & 7) * 2;
    uint8_t* base = out + img * per_chunk * 4;
    *reinterpret_cast<__nv_bfloat16*>(base + off) = hi;
    *reinterpret_cast<__nv_bfloat16*>(base + per_chunk * 2 + off) = lo;
  }
}

struct DenseTcRowsParams {
  const float* A;        // [M, K], leading dimension lda
  const uint8_t* wpack;  // images [n_tile][k_chunk][hi | lo]
  const float* bias;     // [Nout] or null
  float* out;            // [M, Nout], leading dimension ldo
  int M, K, Nout, lda, ldo, NT, n_tiles, n_chunks, act, direct;
};

struct DtSmem {
  int a_off, b_off, t_off, bar_off, total, b_stage;
};
__host__ __device__ inline DtSmem dt_layout(int NT, int with_tbuf) {
  DtSmem l;
  l.b_stage = NT * kDtKc * 4;
  l.a_off = 0;
  l.b_off = kDtStages * kDtAStage;
  l.t_off = l.b_off + kDtStages * l.b_stage;
  l.bar_off = l.t_off + (with_tbuf ? 4 * 32 * 17 * 4 : 0);
  l.bar_off = (l.bar_off + 15) / 16 * 16;
  l.total = l.bar_off + 256;
  return l;
}

__device__ __forceinline__ bool dt_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// [16 rows x 32 columns] fp32 block of a row-major matrix -> registers (one 128-byte request per row, all 16 in flight),
// and registers -> bf16 hi/lo words of a K-major image whose UMMA rows are the matrix ROWS and whose reduction index is
// the matrix COLUMN (rows kernel: A = X tile).  A lane pair (k even, k+1) exchanges values so that the even lane stores
// the packed hi word and the odd lane the packed lo word.
__device__ __forceinline__ void dt_load_rows16(float (&v)[16], const float* __restrict__ src, int ld, int row0,
                                               int n_rows_valid, int col0, int n_cols_valid, int lane) {
#pragma unroll
  for (int j = 0; j < 16; ++j)
    v[j] = (j < n_rows_valid && lane < n_cols_valid) ? __ldg(src + (int64_t)(row0 + j) * ld + col0 + lane) : 0.f;
}
__device__ __forceinline__ void dt_store_rows16(const float (&v)[16], uint8_t* img_hi, uint8_t* img_lo, int img_row0,
                                                int lane) {
  const bool even = (lane & 1) == 0;
  const int kk = lane & ~1;
  uint8_t* img = even ? img_hi : img_lo;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float other = __shfl_xor_sync(0xffffffffu, v[j], 1);
    const float a = even ? v[j] : other, b = even ? other : v[j];
    uint32_t hi, lo;
    tc::split_bf16x2(a, b, hi, lo);
    const int r_img = img_row0 + j;
    const int off = (kk >> 3) * 2048 + (r_img >> 3) * 128 + (r_img & 7) * 16 + (kk & 7) * 2;
    *reinterpret_cast<uint32_t*>(img + off) = even ? hi : lo;
  }
}

__global__ void __launch_bounds__(kDtThreads, 1) dense_tc_rows_kernel(const __grid_constant__ DenseTcRowsParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const DtSmem lay = dt_layout(p.NT, 1);
  uint8_t* smem_a = smem + lay.a_off;
  uint8_t* smem_b = smem + lay.b_off;
  float* tbuf = reinterpret_cast<float*>(smem + lay.t_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* full_a = bars;                 // [stage] 8 producer warps
  uint64_t* full_b = bars + 4;             // [stage] bulk copy (tx)
  uint64_t* empty = bars + 8;              // [stage] tcgen05.commit
  uint64_t* acc_full = bars + 12;          // [buf]   commit
  uint64_t* acc_empty = bars + 14;         // [buf]   4 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_mtiles = (p.M + 127) / 128;
  const int n_items = n_mtiles * p.n_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kDtStages; ++s) {
      tc::mbar_init(&full_a[s], 8);
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&acc_full[b], 1);
      tc::mbar_init(&acc_empty[b], 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == 12) tc::tmem_alloc(tmem_slot, 512);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // ============================ A producers: fp32 rows -> bf16 hi/lo images =============================
    // warp w converts rows [16w, 16w + 16) of the tile.  The loads of the NEXT (item, chunk) are issued before this
    // chunk's barrier wait and conversion: 8 warps x 16-32 requests of 128 bytes keep 16-32 KB in flight per SM
    // (the first version had 4 warps x 8: a third of the latency-bandwidth product, 150 us per launch at 65 536 rows).
    uint32_t it = 0;
    float cur[16], nxt[16];
    int item = blockIdx.x, c = 0;
    if (item < n_items) {
      const int row0 = (item / p.n_tiles) * 128 + warp * 16;
      dt_load_rows16(cur, p.A, p.lda, row0, p.M - row0, 0, p.K, lane);
    }
    while (item < n_items) {
      int n_item = item, n_c = c + 1;
      if (n_c == p.n_chunks) { n_c = 0; n_item = item + gridDim.x; }
      if (n_item < n_items) {
        const int row0 = (n_item / p.n_tiles) * 128 + warp * 16;
        dt_load_rows16(nxt, p.A, p.lda, row0, p.M - row0, n_c * kDtKc, p.K - n_c * kDtKc, lane);
      }
      const uint32_t s = it % kDtStages, ph = (it / kDtStages) & 1;
      ++it;
      tc::mbar_wait(&empty[s], ph ^ 1);
      uint8_t* a_stage = smem_a + s * kDtAStage;
      dt_store_rows16(cur, a_stage, a_stage + kDtAImg, warp * 16, lane);
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&full_a[s]);
#pragma unroll
      for (int j = 0; j < 16; ++j) cur[j] = nxt[j];
      item = n_item;
      c = n_c;
    }
  } else if (warp < 12) {
    // ============================ epilogue: TMEM -> bias / act -> out ======================================
    const int q = warp & 3;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    float* tb = tbuf + q * 32 * 17;
    uint32_t cnt = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++cnt) {
      const int mt = item / p.n_tiles, nt = item - mt * p.n_tiles;
      const uint32_t buf = cnt & 1, par = (cnt >> 1) & 1;
      tc::mbar_wait(&acc_full[buf], par);
      tc::fence_after_thread_sync();
      const int row_base = mt * 128 + q * 32;
      const int n0 = nt * p.NT;
      if (p.direct) {
        // lane = output row: 32 accumulator columns per read, written as 8 float4 of the lane's own 128-byte line
        // (no shared-memory transpose; the sectors of a line are completed by consecutive stores of the same lane)
        const int grow = row_base + lane;
        for (int cb = 0; cb * 32 < p.NT; ++cb) {
          const int col0 = n0 + cb * 32;
          if (col0 >= p.Nout) break;                             // warp-uniform
          const bool second = cb * 32 + 16 < p.NT && col0 + 16 < p.Nout;
          uint32_t v[2][16];
          tc::tmem_ld16(tmem_base + lane_base + buf * kDtMaxNT + cb * 32, v[0]);
          if (second) tc::tmem_ld16(tmem_base + lane_base + buf * kDtMaxNT + cb * 32 + 16, v[1]);
          tc::tmem_wait_ld();
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (h == 1 && !second) break;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const int col = col0 + h * 16 + g * 4;
              if (col >= p.Nout) break;                          // Nout % 4 == 0 on this path
              float4 o = make_float4(__uint_as_float(v[h][4 * g]), __uint_as_float(v[h][4 * g + 1]),
                                     __uint_as_float(v[h][4 * g + 2]), __uint_as_float(v[h][4 * g + 3]));
              if (p.bias) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + col));
                o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
              }
              if (p.act == DTB_ACT_RELU) {
                o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
              } else if (p.act == DTB_ACT_TANH) {
                o.x = tanhf(o.x); o.y = tanhf(o.y); o.z = tanhf(o.z); o.w = tanhf(o.w);
              }
              if (grow < p.M) *reinterpret_cast<float4*>(p.out + (int64_t)grow * p.ldo + col) = o;
            }
          }
        }
      } else
      for (int cb = 0; cb * 16 < p.NT; ++cb) {
        const int col0 = n0 + cb * 16;
        if (col0 >= p.Nout) break;                               // warp-uniform
        uint32_t v[16];
        tc::tmem_ld16(tmem_base + lane_base + buf * kDtMaxNT + cb * 16, v);
        tc::tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float val = __uint_as_float(v[j]);
          if (p.bias && col0 + j < p.Nout) val += __ldg(p.bias + col0 + j);
          if (p.act == DTB_ACT_RELU) val = fmaxf(val, 0.f);
          else if (p.act == DTB_ACT_TANH) val = tanhf(val);
          tb[lane * 17 + j] = val;
        }
        __syncwarp();
        const int col = lane & 15, hrow = lane >> 4;
#pragma unroll
        for (int rr = 0; rr < 16; ++rr) {
          const int r = rr * 2 + hrow;
          const int grow = row_base + r;
          if (grow < p.M && col0 + col < p.Nout) p.out[(int64_t)grow * p.ldo + col0 + col] = tb[r * 17 + col];
        }
        __syncwarp();
      }
      tc::fence_before_thread_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&acc_empty[buf]);
    }
  } else if (warp == 12) {
    // ============================ MMA issue ==================================================================
    const bool leader = dt_elect_one();
    const uint32_t a_u32 = tc::smem_u32(smem_a), b_u32 = tc::smem_u32(smem_b);
    const uint32_t idesc = tc::make_idesc_bf16(128, (uint32_t)p.NT);
    const uint32_t lbo_b = (uint32_t)(p.NT >> 3) * 128;
    const uint32_t img_b = (uint32_t)p.NT * kDtKc * 2;
    uint32_t it = 0, cnt = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++cnt) {
      const uint32_t buf = cnt & 1, par = (cnt >> 1) & 1;
      tc::mbar_wait(&acc_empty[buf], par ^ 1);
      tc::fence_after_thread_sync();
      const uint32_t d_tmem = tmem_base + buf * kDtMaxNT;
      for (int c = 0; c < p.n_chunks; ++c, ++it) {
        const uint32_t s = it % kDtStages, ph = (it / kDtStages) & 1;
        tc::mbar_wait(&full_b[s], ph);
        tc::mbar_wait(&full_a[s], ph);
        tc::fence_after_thread_sync();
        if (leader) {
          const uint32_t a_addr = a_u32 + s * kDtAStage, b_addr = b_u32 + s * (uint32_t)lay.b_stage;
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            // pass 0: A_hi*B_hi ; 1: A_lo*B_hi ; 2: A_hi*B_lo
            const uint32_t a_img = a_addr + (pass == 1 ? kDtAImg : 0);
            const uint32_t b_img = b_addr + (pass == 2 ? img_b : 0);
#pragma unroll
            for (int ks = 0; ks < kDtKc / 16; ++ks) {
              const uint64_t da = tc::make_smem_desc(a_img + ks * 4096, 2048, 128);
              const uint64_t db = tc::make_smem_desc(b_img + ks * 2 * lbo_b, lbo_b, 128);
              tc::mma_ss(d_tmem, da, db, idesc, (uint32_t)((c | pass | ks) != 0));
            }
          }
          tc::mma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (leader) tc::mma_commit(&acc_full[buf]);
      __syncwarp();
    }
  } else {
    // ============================ weight loader ==============================================================
    if (lane == 0) {
      uint32_t it = 0;
      const uint32_t bytes = (uint32_t)lay.b_stage;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int mt = item / p.n_tiles, nt = item - mt * p.n_tiles;
        const uint8_t* src = p.wpack + (size_t)nt * p.n_chunks * bytes;
        for (int c = 0; c < p.n_chunks; ++c, ++it) {
          const uint32_t s = it % kDtStages, ph = (it / kDtStages) & 1;
          tc::mbar_wait(&empty[s], ph ^ 1);
          tc::mbar_arrive_expect_tx(&full_b[s], bytes);
          tc::bulk_g2s(smem_b + (size_t)s * bytes, src + (size_t)c * bytes, bytes, &full_b[s]);
        }
      }
    }
    __syncwarp();
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 12) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------
// weight gradient: dW[k, n] += sum_m X[m, k] dZ[m, n].   UMMA M = 128 in-dim indices k (grid.x), N = NT out-dim indices
// (grid.z), reduction over batch rows in chunks of 32 (grid.y splits the batch).  Both operands are fp32 row-major
// matrices whose ROWS are the reduction index: a lane reads the same column of two consecutive rows (coalesced across
// the warp) and packs the pair into one K-major word.
// ------------------------------------------------------------------------------------------
struct DenseTcWgradParams {
  const float* X;     // [M, K]  ldx
  const float* dZ;    // [M, N]  ldz
  float* dW;          // [K, N]  ldw, accumulated
  float* dbias;       // [N] accumulated by the k-tile-0 CTAs (or null)
  int M, K, N, ldx, ldz, ldw, NT, chunks_per_split, n_chunks_total;
};

// rows [m0, m0+32) x 4 column groups of 32 of src -> K-major image with UMMA row = column index, reduction index = row;
// this warp handles row pairs [pair0, pair0 + 4).  All 32 requests (4 groups x 4 pairs x 2 rows) are issued before the
// first conversion.  Adds the column sums of the values it touched to colsum[] (for the bias gradient).
__device__ __forceinline__ void dt_convert_cols4(const float* __restrict__ src, int ld, int m0, int m_valid, int col0,
                                                 int n_cols, uint8_t* img_hi, uint8_t* img_lo, int img_row0, int img_rows,
                                                 int pair0, int lane, float (&colsum)[4]) {
  float a[4][4], b[4][4];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const bool cok = col0 + g * 32 + lane < n_cols;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int mm = (pair0 + j) * 2;
      a[g][j] = (cok && mm < m_valid) ? __ldg(src + (int64_t)(m0 + mm) * ld + col0 + g * 32 + lane) : 0.f;
      b[g][j] = (cok && mm + 1 < m_valid) ? __ldg(src + (int64_t)(m0 + mm + 1) * ld + col0 + g * 32 + lane) : 0.f;
    }
  }
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int r_img = img_row0 + g * 32 + lane;
    const int base = (r_img >> 3) * 128 + (r_img & 7) * 16;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int mm = (pair0 + j) * 2;
      uint32_t hi, lo;
      tc::split_bf16x2(a[g][j], b[g][j], hi, lo);
      const int off = (mm >> 3) * (img_rows >> 3) * 128 + base + (mm & 7) * 2;
      if (r_img < img_rows) {                     // NT is a multiple of 16, the column groups of 32: the tail group is half used
        *reinterpret_cast<uint32_t*>(img_hi + off) = hi;
        *reinterpret_cast<uint32_t*>(img_lo + off) = lo;
      }
      colsum[g] += a[g][j] + b[g][j];
    }
  }
}

__global__ void __launch_bounds__(kDtWgThreads, 1) dense_tc_wgrad_kernel(const __grid_constant__ DenseTcWgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const DtSmem lay = dt_layout(p.NT, 0);
  uint8_t* smem_a = smem + lay.a_off;
  uint8_t* smem_b = smem + lay.b_off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* full = bars;                   // [stage] 8 producer warps
  uint64_t* empty = bars + 4;              // [stage] commit
  uint64_t* acc_done = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k0 = blockIdx.x * 128, n0 = blockIdx.z * p.NT;
  const int c_begin = blockIdx.y * p.chunks_per_split;
  int c_end = c_begin + p.chunks_per_split;
  if (c_end > p.n_chunks_total) c_end = p.n_chunks_total;
  const int n_ch = c_end > c_begin ? c_end - c_begin : 0;
  const int b_img_bytes = p.NT * kDtKc * 2;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kDtStages; ++s) {
      tc::mbar_init(&full[s], 8);
      tc::mbar_init(&empty[s], 1);
    }
    tc::mbar_init(acc_done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 8) tc::tmem_alloc(tmem_slot, 256);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // warps 0-3: X -> A images (UMMA rows = k);  warps 4-7: dZ -> B images (UMMA rows = n); each warp owns 4 row pairs
    const bool is_a = warp < 4;
    const int pair0 = (warp & 3) * 4;
    float bsum[kDtMaxNT / 32];
#pragma unroll
    for (int g = 0; g < kDtMaxNT / 32; ++g) bsum[g] = 0.f;
    for (int c = 0; c < n_ch; ++c) {
      const uint32_t s = c % kDtStages, ph = (c / kDtStages) & 1;
      tc::mbar_wait(&empty[s], ph ^ 1);
      const int m0 = (c_begin + c) * kDtKc;
      const int m_valid = p.M - m0;
      if (is_a) {
        uint8_t* st = smem_a + s * kDtAStage;
        float unused[4] = {0.f, 0.f, 0.f, 0.f};
        dt_convert_cols4(p.X, p.ldx, m0, m_valid, k0, p.K, st, st + kDtAImg, 0, 128, pair0, lane, unused);
      } else {
        uint8_t* st = smem_b + s * lay.b_stage;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          if (half * 128 < p.NT) {
            float cs[4] = {0.f, 0.f, 0.f, 0.f};
            dt_convert_cols4(p.dZ, p.ldz, m0, m_valid, n0 + half * 128, p.N, st, st + b_img_bytes, half * 128, p.NT, pair0, lane,
                             cs);
#pragma unroll
            for (int g = 0; g < 4; ++g) bsum[half * 4 + g] += cs[g];
          }
        }
      }
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&full[s]);
    }
    if (!is_a && p.dbias && blockIdx.x == 0) {
#pragma unroll
      for (int g = 0; g < kDtMaxNT / 32; ++g) {
        const int n = n0 + g * 32 + lane;
        if (g * 32 < p.NT && n < p.N && bsum[g] != 0.f) atomicAdd(p.dbias + n, bsum[g]);
      }
    }
    // ---- epilogue (warps 0-3, TMEM lane quadrant = warp): accumulator row = k -> dW[k, n0 ...] -----------------
    if (is_a && n_ch > 0) {
      tc::mbar_wait(acc_done, 0);
      tc::fence_after_thread_sync();
      const int k = k0 + warp * 32 + lane;
      const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
      for (int cb = 0; cb * 16 < p.NT; ++cb) {
        if (n0 + cb * 16 >= p.N) break;
        uint32_t v[16];
        tc::tmem_ld16(tmem_base + lane_base + cb * 16, v);
        tc::tmem_wait_ld();
        if (k < p.K) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = n0 + cb * 16 + j;
            if (n < p.N) atomicAdd(p.dW + (int64_t)k * p.ldw + n, __uint_as_float(v[j]));
          }
        }
      }
      tc::fence_before_thread_sync();
    }
  } else if (warp == 8) {
    const bool leader = dt_elect_one();
    const uint32_t a_u32 = tc::smem_u32(smem_a), b_u32 = tc::smem_u32(smem_b);
    const uint32_t idesc = tc::make_idesc_bf16(128, (uint32_t)p.NT);
    const uint32_t lbo_b = (uint32_t)(p.NT >> 3) * 128;
    for (int c = 0; c < n_ch; ++c) {
      const uint32_t s = c % kDtStages, ph = (c / kDtStages) & 1;
      tc::mbar_wait(&full[s], ph);
      tc::fence_after_thread_sync();
      if (leader) {
        const uint32_t a_addr = a_u32 + s * kDtAStage, b_addr = b_u32 + s * (uint32_t)lay.b_stage;
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t a_img = a_addr + (pass == 1 ? kDtAImg : 0);
          const uint32_t b_img = b_addr + (pass == 2 ? (uint32_t)b_img_bytes : 0);
#pragma unroll
          for (int ks = 0; ks < kDtKc / 16; ++ks) {
            const uint64_t da = tc::make_smem_desc(a_img + ks * 4096, 2048, 128);
            const uint64_t db = tc::make_smem_desc(b_img + ks * 2 * lbo_b, lbo_b, 128);
            tc::mma_ss(tmem_base, da, db, idesc, (uint32_t)((c | pass | ks) != 0));
          }
        }
        tc::mma_commit(&empty[s]);
        if (c == n_ch - 1) tc::mma_commit(acc_done);
      }
      __syncwarp();
    }
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 8) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, 256);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct DtTiling {
  int NT, n_tiles, n_chunks;
};
static DtTiling dt_tiling(int K, int Nout) {
  DtTiling t;
  const int np = dt_round_up(Nout, 16);
  t.n_tiles = (np + kDtMaxNT - 1) / kDtMaxNT;
  t.NT = dt_round_up((np + t.n_tiles - 1) / t.n_tiles, 16);
  t.n_chunks = (K + kDtKc - 1) / kDtKc;
  return t;
}

size_t dense_tc_pack_bytes(int K, int Nout) {
  const DtTiling t = dt_tiling(K, Nout);
  return (size_t)t.n_tiles * t.n_chunks * t.NT * kDtKc * 4 + 256;
}

int dense_tc_rows(const float* A, int lda, const float* W, int ldw, int transposed, const float* bias, float* out,
                  int ldo, int M, int K, int Nout, int act, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (M <= 0) return DTB_OK;
  if (!workspace || workspace_bytes < dense_tc_pack_bytes(K, Nout) || (reinterpret_cast<uintptr_t>(workspace) & 15)) {
    set_error("dense_tc_rows: workspace missing, misaligned or smaller than the packed weights (%zu bytes needed)",
              dense_tc_pack_bytes(K, Nout));
    return DTB_ERR_INVALID_ARG;
  }
  const DtTiling t = dt_tiling(K, Nout);
  const int64_t total = (int64_t)t.n_tiles * t.n_chunks * t.NT * kDtKc;
  int blocks = (int)((total + 255) / 256);
  if (blocks > sm_count() * 4) blocks = sm_count() * 4;
  dense_tc_pack_kernel<<<blocks, 256, 0, st>>>(W, reinterpret_cast<uint8_t*>(workspace), K, Nout, ldw, t.NT, t.n_tiles,
                                               t.n_chunks, transposed);
  DTB_LAUNCH_OK();
  DenseTcRowsParams p{};
  p.A = A; p.wpack = reinterpret_cast<const uint8_t*>(workspace); p.bias = bias; p.out = out;
  p.M = M; p.K = K; p.Nout = Nout; p.lda = lda; p.ldo = ldo; p.NT = t.NT; p.n_tiles = t.n_tiles; p.n_chunks = t.n_chunks;
  p.act = act;
  p.direct = (Nout % 4 == 0 && ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
              (!bias || (reinterpret_cast<uintptr_t>(bias) & 15) == 0)) ? 1 : 0;
  const DtSmem lay = dt_layout(t.NT, 1);
  DTB_CUDA_OK(cudaFuncSetAttribute(dense_tc_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lay.total));
  const int n_items = ((M + 127) / 128) * t.n_tiles;
  int grid = sm_count();
  if (grid > n_items) grid = n_items;
  dense_tc_rows_kernel<<<grid, kDtThreads, lay.total, st>>>(p);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int dense_tc_wgrad(const float* X, int ldx, const float* dZ, int ldz, float* dW, int ldw, float* dbias, int M, int K,
                   int N, cudaStream_t st) {
  if (M <= 0) return DTB_OK;
  DenseTcWgradParams p{};
  const int np = dt_round_up(N, 16);
  const int n_tiles = (np + kDtMaxNT - 1) / kDtMaxNT;
  p.NT = dt_round_up((np + n_tiles - 1) / n_tiles, 16);
  p.X = X; p.dZ = dZ; p.dW = dW; p.dbias = dbias;
  p.M = M; p.K = K; p.N = N; p.ldx = ldx; p.ldz = ldz; p.ldw = ldw;
  p.n_chunks_total = (M + kDtKc - 1) / kDtKc;
  const int k_tiles = (K + 127) / 128;
  int splits = sm_count() / (k_tiles * n_tiles);
  if (splits < 1) splits = 1;
  if (splits > p.n_chunks_total) splits = p.n_chunks_total;
  p.chunks_per_split = (p.n_chunks_total + splits - 1) / splits;
  splits = (p.n_chunks_total + p.chunks_per_split - 1) / p.chunks_per_split;
  const DtSmem lay = dt_layout(p.NT, 0);
  DTB_CUDA_OK(cudaFuncSetAttribute(dense_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lay.total));
  dense_tc_wgrad_kernel<<<dim3(k_tiles, splits, n_tiles), kDtWgThreads, lay.total, st>>>(p);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

}  // namespace dtb
