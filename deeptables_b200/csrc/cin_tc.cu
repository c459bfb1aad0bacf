// CIN (layers.py:638-734) on the 5th-generation tensor cores -- the product path.
//
// Math.  For batch row b, embedding dim d:  C_k[(b,d), l] = sum_{i,j} x0[b,i,d] h_k[b,j,d] W_k[i*H+j, l].
// That is a GEMM whose A operand  Z_k[(b,d), (i,j)] = x0[b,i,d]*h_k[b,j,d]  never needs to exist in
// HBM (the reference materialises it: 7 GB per layer at B = 65 536, layers.py:693-695).  Here one CTA
// owns 2 x (128/D) batch rows = two M=128 tiles; thread p of a tile's producer group owns GEMM row
// m = p = (row r, dim d), keeps h_k[b, :, d] in REGISTERS across the whole layer (it is that thread's
// own slice of the previous accumulator), and per K-chunk (one x0 field i, all j) multiplies by the
// scalar x0[b,i,d], splits the fp32 products into bf16 hi + lo and hands them to the tensor core
// through TMEM (tcgen05.st, A-from-TMEM MMA).  W_k is pre-split into bf16 hi/lo and pre-tiled in the
// UMMA canonical layout by a tiny pack kernel, so a whole K-chunk (<= 32 KB) arrives with ONE bulk
// async copy.
//
// Precision.  bf16x3: Z_hi*W_hi + Z_lo*W_hi + Z_hi*W_lo, fp32 accumulate in TMEM: relative error
// ~2^-16 per product -- inside the 1e-3 parity bar with margin (single-pass bf16 is ~4e-3).
//
// Pipeline per CTA (320 threads): warps 0-3 / 4-7 = producer+epilogue groups of tile 0 / 1 (warp%4 =
// TMEM lane quadrant), warp 8 = MMA issuer (one thread) + TMEM allocator, warp 9 = weight loader.
// mbarriers: full_a[tile][stage] (producers -> MMA), full_b[stage] (bulk copy -> MMA),
// empty_a / empty_b (tcgen05.commit -> producers / loader), acc_full[tile] (commit -> epilogue).
// Both tiles share each W chunk in smem, which halves the L2->SM weight stream (the limiter at one
// tile per CTA: 42 B/clk/SM against a ~42 B/clk/SM L2 cap).
#include "dtb_common.cuh"
#include "cin_impl.h"
#include "tcgen05.cuh"
#include "cin_tc_common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace dtb {

// ------------------------------------------------------------------------------------------
// weight pack: fp32 [K_k, L_k] -> per chunk i: [hi image | lo image], image = canonical K-major
// no-swizzle tile of B[n][kk] = W[(i*H + kk), n]  (zero for kk >= H): core (kk/8, n/8) at
// ((kk/8)*(L/8) + n/8)*128 B, row n%8 at 16 B, element kk%8 at 2 B.
// ------------------------------------------------------------------------------------------
__global__ void cin_tc_pack_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int F, int H, int Hp,
                                   int L) {
  const int64_t per_chunk = (int64_t)L * Hp;
  const int64_t total = per_chunk * F;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(t / per_chunk);
    const int rem = (int)(t - (int64_t)i * per_chunk);
    const int kk = rem / L, n = rem - kk * L;     // n fastest: coalesced reads of W rows
    const float v = kk < H ? w[((int64_t)i * H + kk) * L + n] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    const int64_t off = ((int64_t)(kk >> 3) * (L >> 3) + (n >> 3)) * 128 + (n & 7) * 16 + (kk & 7) * 2;
    uint8_t* base = out + (int64_t)i * per_chunk * 4;      // hi + lo images, 2 bytes each
    *reinterpret_cast<__nv_bfloat16*>(base + off) = hi;
    *reinterpret_cast<__nv_bfloat16*>(base + per_chunk * 2 + off) = lo;
  }
}

// ------------------------------------------------------------------------------------------
// forward kernel
// ------------------------------------------------------------------------------------------
// A pipeline granule ("sub-chunk") = one x0 field i x 32 hidden fields j = two K=16 UMMA steps.
// A operand of a granule in TMEM: 16 columns hi + 16 columns lo per tile; kStagesA granules x 2 tiles
// in flight = 256 columns, next to the two 128-column accumulators.  The weight chunk of field i (all
// Hp hidden fields, hi+lo, <= 32 KB) is one bulk copy and serves both tiles and both granules.
// ---- single-pass fp16 kernels (cin_tc2.cu): max|W_k| (bit pattern, atomicMax on the int view of non-negative floats) and the scaled pack
__global__ void cin_tc_wmax_kernel(const float* __restrict__ w, int64_t n, int* __restrict__ out) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float a = fabsf(w[i]);
    if (a < __int_as_float(0x7f800000)) m = fmaxf(m, a);      // ignore inf / nan
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_int(m));
}

// same image layout as cin_tc_pack_kernel, but ONE fp16 image per chunk (the "hi" slot), values scaled by the
// power of two that brings max|W_k| into [2^9, 2^10)
__global__ void cin_tc_pack_f16_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int F, int H, int Hp,
                                       int L, const int* __restrict__ wmax) {
  float s, inv;
  tc::pow2_scale_to_1024(__int_as_float(*wmax), s, inv);
  const int64_t per_chunk = (int64_t)L * Hp;
  const int64_t total = per_chunk * F;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(t / per_chunk);
    const int rem = (int)(t - (int64_t)i * per_chunk);
    const int kk = rem / L, n = rem - kk * L;       // n fastest: coalesced reads
    const float v = kk < H ? w[((int64_t)i * H + kk) * L + n] * s : 0.f;
    const int64_t off = ((int64_t)(kk >> 3) * (L >> 3) + (n >> 3)) * 128 + (n & 7) * 16 + (kk & 7) * 2;
    *reinterpret_cast<__half*>(out + (int64_t)i * per_chunk * 4 + off) = __float2half_rn(v);
  }
}

struct TcSmemLayout {
  int b_off, x0_off, bar_off, total;
};

__host__ __device__ inline TcSmemLayout tc_layout(int b_stage_bytes, int F) {
  TcSmemLayout l;
  l.b_off = 0;
  l.x0_off = kStagesB * b_stage_bytes;
  l.bar_off = l.x0_off + 2 * 128 * F * 4;          // x0s[tile][r][i][d]
  l.bar_off = (l.bar_off + 15) / 16 * 16;
  l.total = l.bar_off + 256;
  return l;
}

template <int D>
__global__ void __launch_bounds__(kTcThreads, 1) cin_tc_fwd_kernel(const __grid_constant__ CinTcParams p) {
  constexpr int R = 128 / D;                 // batch rows per M=128 tile
  extern __shared__ __align__(1024) uint8_t smem[];
  const TcSmemLayout lay = tc_layout(p.b_stage_bytes, p.F);
  uint8_t* smem_b = smem + lay.b_off;
  float* x0s = reinterpret_cast<float*>(smem + lay.x0_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* full_a = bars;                        // [tile][stage] -> 8
  uint64_t* empty_a = bars + 8;                   // [stage]       -> 4
  uint64_t* full_b = bars + 12;                   // [stage]       -> 4
  uint64_t* empty_b = bars + 16;                  // [stage]       -> 4
  uint64_t* acc_full = bars + 20;                 // [tile]        -> 2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = p.F;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2 * kStagesA; ++i) tc::mbar_init(&full_a[i], 4);   // one arrival per producer warp
    for (int s = 0; s < kStagesA; ++s) tc::mbar_init(&empty_a[s], 1);
    for (int s = 0; s < kStagesB; ++s) {
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty_b[s], 1);
    }
    tc::mbar_init(&acc_full[0], 1);
    tc::mbar_init(&acc_full[1], 1);
    tc::fence_barrier_init();
  }
  if (warp == 8) tc::tmem_alloc(tmem_slot, kTmemCols);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // =================== producer + epilogue group g, GEMM row m = t =========================
    const int g = warp >> 2;
    const int t = threadIdx.x & 127;
    const int r = t / D, d = t % D;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    float* x0g = x0s + (size_t)g * 128 * F;         // [r][i][d]
    uint32_t gran = 0, layer_cnt = 0;
    float h[kMaxHp];
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      const int row0 = (st * 2 + g) * R;
      const int b = row0 + r;
      // ---- gather this tile's x0 block: R rows x F fields x D floats, 16-byte pieces ----------
      {
        constexpr int Q = D / 4;
        for (int e = t; e < R * F * Q; e += 128) {
          const int rr = e / (F * Q);
          const int rem = e - rr * F * Q;
          const int i = rem / Q, q = rem - i * Q;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row0 + rr < p.B) {
            const int64_t rb = table_row(p.row_offsets, i, __ldg(p.idx + (int64_t)(row0 + rr) * F + i), D, p.status);
            if (rb >= 0) v = ldg_stream_f4(p.table + rb + (q << 2));
          }
          *reinterpret_cast<float4*>(x0g + ((size_t)rr * F + i) * D + (q << 2)) = v;
        }
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
      // ---- h_0 = x0 (zero padded to Hp[0]) ; training: save x0t ------------------------------
#pragma unroll
      for (int j = 0; j < kMaxHp; ++j) h[j] = (j < F) ? x0g[((size_t)r * F + j) * D + d] : 0.f;
      if (p.saved) {
        if (b < p.B && !p.compact) {
          float* dst = p.saved + ((size_t)b * D + d) * F;
          for (int j = 0; j < F; ++j) dst[j] = x0g[((size_t)r * F + j) * D + d];
        }
        // block-transposed copy for the wgrad kernel: [m / 64][field][68] (rows of a 64-row stage contiguous
        // along m, padded to 68 floats so LDS.128 across fields is conflict-free); padded rows get zeros
        const size_t m_pad = (size_t)(st * 2 + g) * 128 + t;
        float* xb = p.saved + p.xb_off + (m_pad >> 6) * (size_t)(F * kWgPad) + (m_pad & 63);
        for (int j = 0; j < F; ++j) xb[j * kWgPad] = x0g[((size_t)r * F + j) * D + d];
      }
      for (int k = 0; k < p.n_layers; ++k) {
        const int Hp = p.Hp[k], L = p.L[k];
        for (int i = 0; i < F; ++i) {
          const float xi = x0g[((size_t)r * F + i) * D + d];
#pragma unroll
          for (int half = 0; half < kMaxHp / kSubK; ++half) {
            if (half * kSubK < Hp) {
              const uint32_t sa = gran % kStagesA, pa = (gran / kStagesA) & 1;
              ++gran;
              // 32 products of this granule -> packed bf16x2 hi / lo (all computed before the async
              // tcgen05.st are issued, so every store reads registers of its own)
              uint32_t zh[kACols], zl[kACols];
#pragma unroll
              for (int q = 0; q < kACols; ++q)
                tc::split_bf16x2(xi * h[half * kSubK + 2 * q], xi * h[half * kSubK + 2 * q + 1], zh[q], zl[q]);
              tc::mbar_wait(&empty_a[sa], pa ^ 1);
              tc::fence_after_thread_sync();
              const uint32_t a_col = tmem_base + lane_base + 2 * kAccCols + ((sa * 2 + g) * 2) * kACols;
              tc::tmem_st8v(a_col, zh[0], zh[1], zh[2], zh[3], zh[4], zh[5], zh[6], zh[7]);
              tc::tmem_st8v(a_col + 8, zh[8], zh[9], zh[10], zh[11], zh[12], zh[13], zh[14], zh[15]);
              if (p.n_pass > 1) {
                tc::tmem_st8v(a_col + kACols, zl[0], zl[1], zl[2], zl[3], zl[4], zl[5], zl[6], zl[7]);
                tc::tmem_st8v(a_col + kACols + 8, zl[8], zl[9], zl[10], zl[11], zl[12], zl[13], zl[14], zl[15]);
              }
              tc::tmem_wait_st();
              tc::fence_before_thread_sync();
              __syncwarp();
              if (lane == 0) tc::mbar_arrive(&full_a[g * kStagesA + sa]);
            }
          }
        }
        // ---- epilogue of layer k: this thread's accumulator row -> bias/act -> h / pooled / saved
        tc::mbar_wait(&acc_full[g], layer_cnt & 1);
        ++layer_cnt;
        tc::fence_after_thread_sync();
        const int hid_n = p.hid_n[k], pool_lo = p.pool_lo[k], pool_n = p.pool_n[k];
        const float* bias = p.bias ? p.bias + p.bias_off[k] : nullptr;
        float* sv = (p.saved && !p.compact && b < p.B) ? p.saved + p.saved_off[k] + ((size_t)b * D + d) * L : nullptr;
        // compact format: one bit per feature map (output > 0) at the head of the T_k region, ceil(L/32) words per row
        const int mask_words = (L + 31) >> 5;
        uint32_t* mrow = (p.saved && p.compact && p.act == DTB_ACT_RELU && b < p.B)
                             ? reinterpret_cast<uint32_t*>(p.saved + p.saved_off[k]) + ((size_t)b * D + d) * mask_words
                             : nullptr;
        uint32_t mw[kMaxL / 32];
#pragma unroll
        for (int w = 0; w < kMaxL / 32; ++w) mw[w] = 0u;
        // block-transposed copy of the hidden half for the wgrad kernel ([m / 64][j][68], zeros in padded rows)
        float* hb = nullptr;
        if (p.saved && hid_n > 0) {
          const size_t m_pad = (size_t)(st * 2 + g) * 128 + t;
          hb = p.saved + p.hb_off[k] + (m_pad >> 6) * (size_t)(hid_n * kWgPad) + (m_pad & 63);
        }
#pragma unroll
        for (int cb = 0; cb < kMaxL / 16; ++cb) {
          if (cb * 16 < L) {
            uint32_t v[16];
            tc::tmem_ld16(tmem_base + lane_base + g * kAccCols + cb * 16, v);
            tc::tmem_wait_ld();
            float o[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float val = __uint_as_float(v[j]);
              if (bias) val += __ldg(bias + cb * 16 + j);
              if (p.act == DTB_ACT_RELU) val = fmaxf(val, 0.f);
              o[j] = val;
              if (cb * 16 + j < kMaxHp) {
                if (cb * 16 + j < hid_n) h[cb * 16 + j] = val;
              }
            }
            if (sv) {
#pragma unroll
              for (int j = 0; j < 16; j += 4)
                *reinterpret_cast<float4*>(sv + cb * 16 + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
            }
            {
              uint32_t bits = 0u;
#pragma unroll
              for (int j = 0; j < 16; ++j) bits |= (o[j] > 0.f ? 1u : 0u) << j;
              mw[cb >> 1] |= bits << ((cb & 1) * 16);
            }
            if (hb) {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (cb * 16 + j < hid_n) hb[(cb * 16 + j) * kWgPad] = o[j];     // x0 == 0 for padded rows => o == act(bias): harmless, dC == 0 there
            }
            // sum over the D lanes that share a batch row.  Reduce-scatter butterfly: at offset `off` a
            // lane keeps the half of its live columns selected by its bit `off` and adds the partner's
            // copy of that half, so after log2(D) steps lane d holds the total of column (block + d):
            // D-1 shuffles per D columns instead of D*log2(D), and a coalesced store.
            if constexpr (D <= 16) {
#pragma unroll
              for (int blk = 0; blk < 16 / D; ++blk) {
                const int col0 = cb * 16 + blk * D;
                if (col0 + D > pool_lo && col0 < pool_lo + pool_n) {     // warp-uniform
                  float w[D];
#pragma unroll
                  for (int j = 0; j < D; ++j) w[j] = o[blk * D + j];
#pragma unroll
                  for (int off = D / 2; off >= 1; off >>= 1) {
                    const bool up = (d & off) != 0;
#pragma unroll
                    for (int j = 0; j < off; ++j) {
                      const float send = up ? w[j] : w[j + off];
                      const float keep = up ? w[j + off] : w[j];
                      w[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                    }
                  }
                  const int col = col0 + d;
                  if (b < p.B && col >= pool_lo && col < pool_lo + pool_n)
                    p.pooled[(size_t)b * p.P + p.pcol0[k] + (col - pool_lo)] = w[0];
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const int col = cb * 16 + j;
                if (col >= pool_lo && col < pool_lo + pool_n) {      // warp-uniform
                  float sum = o[j];
#pragma unroll
                  for (int off = 1; off < 32; off <<= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
                  if (d == 0 && b < p.B) p.pooled[(size_t)b * p.P + p.pcol0[k] + (col - pool_lo)] = sum;
                }
              }
            }
          }
        }
        if (mrow) {
#pragma unroll
          for (int w = 0; w < kMaxL / 32; ++w)
            if (w < mask_words) mrow[w] = mw[w];
        }
        // zero the padding of the next layer's K chunk
        if (k + 1 < p.n_layers) {
#pragma unroll
          for (int j = 0; j < kMaxHp; ++j)
            if (j >= hid_n) h[j] = 0.f;
        }
        tc::fence_before_thread_sync();
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");   // x0 block free for the next super tile
    }
  } else if (warp == 8) {
    // ================================ MMA issuer ===============================================
    // The whole warp walks the schedule (warp-uniform values -> uniform registers); one elected lane
    // issues the tcgen05 instructions.
    const bool leader = elect_one_sync();
    const uint32_t smem_b_u32 = tc::smem_u32(smem_b);
    uint32_t gran = 0, chunk = 0;
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      for (int k = 0; k < p.n_layers; ++k) {
        const int Hp = p.Hp[k], L = p.L[k];
        const uint32_t idesc = tc::make_idesc_bf16(128, (uint32_t)L);
        const uint32_t lbo_b = (uint32_t)(L >> 3) * 128;       // K-direction core stride of the W image
        const uint32_t img_b = (uint32_t)L * Hp * 2;           // bytes of one (hi or lo) image
        // static part of the W descriptor: LBO, SBO = 128 B, version 1, no swizzle
        const uint64_t desc_hi = ((uint64_t)((lbo_b >> 4) & 0x3FFF) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
        for (int i = 0; i < F; ++i, ++chunk) {
          const uint32_t sb = chunk % kStagesB, pb = (chunk / kStagesB) & 1;
          tc::mbar_wait(&full_b[sb], pb);
          const uint32_t b_addr = smem_b_u32 + sb * (uint32_t)p.b_stage_bytes;
          for (int half = 0; half * kSubK < Hp; ++half, ++gran) {
            const uint32_t sa = gran % kStagesA, pa = (gran / kStagesA) & 1;
            const bool last = (i == F - 1) && ((half + 1) * kSubK >= Hp);
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              tc::mbar_wait(&full_a[g * kStagesA + sa], pa);
              tc::fence_after_thread_sync();
              if (leader) {
                const uint32_t d_tmem = tmem_base + g * kAccCols;
                const uint32_t a_base = tmem_base + 2 * kAccCols + ((sa * 2 + g) * 2) * kACols;
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                  if (pass < p.n_pass) {
                    // pass 0: A_hi*B_hi ; 1: A_lo*B_hi ; 2: A_hi*B_lo
                    const uint32_t a_addr = a_base + (pass == 1 ? kACols : 0);
                    const uint32_t b_img = b_addr + (pass == 2 ? img_b : 0) + (uint32_t)half * 4 * lbo_b;
#pragma unroll
                    for (int ks = 0; ks < kSubK / 16; ++ks) {
                      const uint32_t acc = (uint32_t)((i | half | pass | ks) != 0);
                      const uint64_t desc_b = desc_hi | (uint64_t)(((b_img + ks * 2 * lbo_b) >> 4) & 0x3FFF);
                      tc::mma_ts(d_tmem, a_addr + ks * 8, desc_b, idesc, acc);
                    }
                  }
                }
                if (last) tc::mma_commit(&acc_full[g]);
              }
              __syncwarp();
            }
            if (leader) tc::mma_commit(&empty_a[sa]);
            __syncwarp();
          }
          if (leader) tc::mma_commit(&empty_b[sb]);
          __syncwarp();
        }
      }
    }
  } else {
    // ================================ weight loader ============================================
    if (lane == 0) {
      uint32_t chunk = 0;
      for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
        for (int k = 0; k < p.n_layers; ++k) {
          const uint32_t bytes = (uint32_t)p.L[k] * p.Hp[k] * 2 * (p.n_pass > 1 ? 2 : 1);
          const uint32_t stride = (uint32_t)p.L[k] * p.Hp[k] * 4;
          const uint8_t* src = p.wpack + p.wpack_off[k];
          for (int i = 0; i < F; ++i, ++chunk) {
            const uint32_t sb = chunk % kStagesB, pb = (chunk / kStagesB) & 1;
            tc::mbar_wait(&empty_b[sb], pb ^ 1);
            tc::mbar_arrive_expect_tx(&full_b[sb], bytes);
            tc::bulk_g2s(smem_b + (size_t)sb * p.b_stage_bytes, src + (size_t)i * stride, bytes, &full_b[sb]);
          }
        }
      }
    }
    __syncwarp();
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 8) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------
// tensor-core self test: C[128,N] = A[128,K] * Bimg^T with single-pass bf16 (isolates descriptor /
// TMEM-layout mistakes from the CIN logic).  Bimg is a packed image from cin_tc_pack_kernel.
// ------------------------------------------------------------------------------------------
template <bool kATmem>
__global__ void __launch_bounds__(160, 1) tc_selftest_kernel(const float* __restrict__ A, const uint8_t* __restrict__ bimg,
                                                              float* __restrict__ C, int N, int K) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smem_b = smem;                                   // N*K*2
  uint8_t* smem_a = smem + 128 * 64 * 2;                    // 128*K*2
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * 128 * 64 * 2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tc::mbar_init(&bars[0], 128);   // full_a
    tc::mbar_init(&bars[1], 1);     // full_b
    tc::mbar_init(&bars[2], 1);     // acc_full
    tc::fence_barrier_init();
  }
  if (warp == 4) tc::tmem_alloc(tmem_slot, 256);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (warp < 4) {
    const int t = threadIdx.x;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    if (t == 0) {
      tc::mbar_arrive_expect_tx(&bars[1], (uint32_t)N * K * 2);
      tc::bulk_g2s(smem_b, bimg, (uint32_t)N * K * 2, &bars[1]);
    }
    for (int jb = 0; jb < K / 16; ++jb) {
      uint32_t hi[8];
      for (int q = 0; q < 8; ++q) hi[q] = tc::pack_bf16x2(A[t * K + jb * 16 + 2 * q], A[t * K + jb * 16 + 2 * q + 1]);
      if constexpr (kATmem) {
        tc::tmem_st8(tmem_base + lane_base + 128 + jb * 8, hi);
      } else {
        const int row_off = (t >> 3) * 128 + (t & 7) * 16;
        *reinterpret_cast<uint4*>(smem_a + (2 * jb) * 2048 + row_off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(smem_a + (2 * jb + 1) * 2048 + row_off) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
      }
    }
    if constexpr (kATmem) {
      tc::tmem_wait_st();
      tc::fence_before_thread_sync();
    } else {
      tc::fence_proxy_async_smem();
    }
    tc::mbar_arrive(&bars[0]);
    tc::mbar_wait(&bars[2], 0);
    tc::fence_after_thread_sync();
    for (int cb = 0; cb < N / 16; ++cb) {
      uint32_t v[16];
      tc::tmem_ld16(tmem_base + lane_base + cb * 16, v);
      tc::tmem_wait_ld();
      for (int j = 0; j < 16; ++j) C[t * N + cb * 16 + j] = __uint_as_float(v[j]);
    }
    tc::fence_before_thread_sync();
  } else if (lane == 0) {
    tc::mbar_wait(&bars[1], 0);
    tc::mbar_wait(&bars[0], 0);
    tc::fence_after_thread_sync();
    const uint32_t idesc = tc::make_idesc_bf16(128, (uint32_t)N);
    const uint32_t lbo_b = (uint32_t)(N >> 3) * 128;
    for (int ks = 0; ks < K / 16; ++ks) {
      const uint64_t desc_b = tc::make_smem_desc(tc::smem_u32(smem_b) + ks * 2 * lbo_b, lbo_b, 128);
      if constexpr (kATmem)
        tc::mma_ts(tmem_base, tmem_base + 128 + ks * 8, desc_b, idesc, ks != 0);
      else
        tc::mma_ss(tmem_base, tc::make_smem_desc(tc::smem_u32(smem_a) + ks * 4096, 2048, 128), desc_b, idesc, ks != 0);
    }
    tc::mma_commit(&bars[2]);
  }
  __syncwarp();
  __syncthreads();
  if (warp == 4) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, 256);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int g_tc_bwd_fp32 = 0;   // test hook (bit 16 of set_variant): run the exact-fp32 backward after the tensor-core forward
static int g_tc_full_save = 0;  // test hook (bit 17 of set_variant): keep the fp32 T_k rows in the saved activations

static bool d_supported(int D) { return D == 4 || D == 8 || D == 16 || D == 32; }
static bool cin_tc_bwd_supported(const CinShape& s);

// Saved-activation format of a training forward.  Full: x0t + fp32 T_k rows (what the exact-fp32 backward reads)
// + the block-transposed operand tiles.  Compact: the tensor-core backward needs only the sign of each output
// (relu mask, 1 bit) and the hidden halves, which the block-transposed tiles already hold -- so T_k shrinks to
// ceil(L/32) words per row and x0t is not written: -1.7 GB of writes in forward and of reads in dgrad at
// B = 65 536.  Both halves of a step evaluate this predicate, so it must not change between them.
static bool cin_tc_compact(const CinShape& s) { return !g_tc_full_save && !g_tc_bwd_fp32 && cin_tc_bwd_supported(s); }

bool cin_tc_supported(const CinShape& s) {
  if (!d_supported(s.D)) return false;
  if (s.F > kMaxHp || s.F < 1) return false;
  for (int k = 0; k < s.n_layers; ++k) {
    if (s.L[k] % 16 || s.L[k] > kMaxL) return false;
    if (round_up(s.H[k], kSubK) > kMaxHp) return false;
    if (k > 0 && s.H[k] % 4) return false;
  }
  // shared-memory budget of the forward kernel
  int bstage = 0;
  for (int k = 0; k < s.n_layers; ++k) {
    const int bytes = 4 * s.L[k] * round_up(s.H[k], kSubK);
    if (bytes > bstage) bstage = bytes;
  }
  return tc_layout(bstage, s.F).total <= 227 * 1024;
}

// precision "auto": the single-pass fp16 kernels of cin_tc2.cu when forward, data gradient and weight gradient all
// support the shape (and the compact saved-activation format is in force), else the bf16x3 kernels of this file
bool cin_tc_f16_auto(const CinShape& s) {
  if (!cin_tc_supported(s) || !cin_tc_compact(s)) return false;
  CinTcParams f{};
  CinTcBwdParams b{};
  f.F = b.F = s.F; f.n_layers = b.n_layers = s.n_layers; f.n_pass = 1; f.compact = b.compact = 1;
  f.saved = reinterpret_cast<float*>(16);       // "training": the stricter of the two forward checks
  for (int k = 0; k < s.n_layers; ++k) {
    f.L[k] = b.L[k] = s.L[k]; f.H[k] = b.H[k] = s.H[k]; f.Hp[k] = b.Hp[k] = round_up(s.H[k], kSubK);
    f.pool_lo[k] = b.pool_lo[k] = s.pool_lo[k]; f.pool_n[k] = b.pool_n[k] = s.pool_n[k];
    f.hid_n[k] = b.hid_n[k] = (k + 1 < s.n_layers) ? s.H[k + 1] : 0;
  }
  return cin_tc2_fwd_supported(f, s.D) && cin_tc2_bwd_supported(b, s.D);
}

static size_t wpack_bytes(const CinShape& s) {
  size_t b = 0;
  for (int k = 0; k < s.n_layers; ++k) b += (size_t)s.F * s.L[k] * round_up(s.H[k], kSubK) * 4;
  return b;
}

// grid of the weight-pack kernels of layer k: one thread per packed element, at most 8 CTAs per SM
static int pack_grid(const CinShape& s, int Hp, int k) {
  const int64_t total = (int64_t)s.F * s.L[k] * Hp;
  int blocks = (int)((total + 255) / 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  return blocks;
}

static size_t m_pad_rows(const CinShape& s, int B) {
  const int R = 128 / s.D;
  return (((size_t)B + 2 * R - 1) / (2 * R)) * 256;
}
static size_t bt_floats(const CinShape& s, int B) {      // block-transposed copies: x0 and h_k (k >= 1)
  const size_t blocks = m_pad_rows(s, B) / 64;
  size_t n = blocks * s.F * kWgPad;
  for (int k = 1; k < s.n_layers; ++k) n += blocks * s.H[k] * kWgPad;
  return n;
}
size_t cin_tc_saved_bytes(const CinShape& s, int B) { return cin_fp32_saved_bytes(s, B) + bt_floats(s, B) * sizeof(float); }

size_t cin_tc_bwd_workspace_bytes(const CinShape& s, int B);
size_t cin_tc_workspace_bytes(const CinShape& s, int B, int training) {
  size_t need = wpack_bytes(s) + 1024;
  if (training) {
    const size_t a = cin_tc_bwd_workspace_bytes(s, B), b = cin_fp32_workspace_bytes(s, B, 1);
    need = need > a ? need : a;
    need = need > b ? need : b;     // the exact-fp32 backward stays selectable (tests, unsupported shapes)
  }
  return need;
}

template <int D>
static int launch_fwd(const CinTcParams& p, int smem_bytes, cudaStream_t st) {
  auto kern = cin_tc_fwd_kernel<D>;
  DTB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  const int R = 128 / D;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);
  int grid = sm_count();
  if (grid > n_super) grid = n_super;
  kern<<<grid, kTcThreads, smem_bytes, st>>>(p);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int cin_tc_fwd(const CinShape& s, const int32_t* idx, const float* table, const int64_t* row_offsets,
               const float* weights, const float* bias, float* pooled, void* saved, void* workspace,
               size_t workspace_bytes, int B, int act, int n_pass, int f16, int* status, cudaStream_t st) {
  if (f16 && workspace_bytes < wpack_bytes(s) + 64) {
    set_error("dtb_cin_fwd: workspace too small for the fp16 weight images and their scale words");
    return DTB_ERR_INVALID_ARG;
  }
  if (workspace_bytes < wpack_bytes(s)) {
    set_error("dtb_cin_fwd: workspace too small for the packed weights");
    return DTB_ERR_INVALID_ARG;
  }
  if ((reinterpret_cast<uintptr_t>(table) % 16) || (reinterpret_cast<uintptr_t>(workspace) % 16)) {
    set_error("dtb_cin_fwd: table / workspace must be 16-byte aligned");
    return DTB_ERR_INVALID_ARG;
  }
  CinTcParams p{};
  p.idx = idx; p.table = table; p.row_offsets = row_offsets;
  p.wpack = reinterpret_cast<uint8_t*>(workspace);
  p.bias = bias; p.pooled = pooled; p.saved = reinterpret_cast<float*>(saved); p.status = status;
  p.B = B; p.F = s.F; p.n_layers = s.n_layers; p.act = act; p.n_pass = n_pass; p.P = s.P;
  size_t woff = 0, soff = (size_t)B * s.D * s.F;
  const size_t bt_blocks = m_pad_rows(s, B) / 64;
  p.xb_off = cin_fp32_saved_bytes(s, B) / sizeof(float);
  size_t hoff = p.xb_off + bt_blocks * s.F * kWgPad;
  int bstage = 0;
  for (int k = 0; k < s.n_layers; ++k) {
    p.L[k] = s.L[k]; p.H[k] = s.H[k]; p.Hp[k] = round_up(s.H[k], kSubK);
    p.pool_lo[k] = s.pool_lo[k]; p.pool_n[k] = s.pool_n[k]; p.pcol0[k] = s.pcol0[k];
    p.hid_n[k] = (k + 1 < s.n_layers) ? s.H[k + 1] : 0;
    p.wpack_off[k] = woff;
    p.saved_off[k] = soff;
    p.hb_off[k] = hoff;
    hoff += bt_blocks * p.hid_n[k] * kWgPad;
    p.bias_off[k] = s.b_off[k];
    const size_t chunk = (size_t)s.L[k] * p.Hp[k] * 4;
    woff += chunk * s.F;
    soff += (size_t)B * s.D * s.L[k];
    if ((int)chunk > bstage) bstage = (int)chunk;
  }
  p.b_stage_bytes = bstage;
  p.compact = cin_tc_compact(s) ? 1 : 0;
  int* wmax = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(workspace) + wpack_bytes(s));     // behind the images
  p.wmax = wmax;
  // the single fp16 pass runs on the two-threads-per-row kernels of cin_tc2.cu only
  if (f16 && !cin_tc2_fwd_supported(p, s.D)) {
    set_error("dtb_cin_fwd: fp16 single pass: shape outside cin_tc2 (F=%d D=%d); use precision 0/2", s.F, s.D);
    return DTB_ERR_UNSUPPORTED;
  }
  for (int k = 0; k < s.n_layers; ++k) {
    uint8_t* img = reinterpret_cast<uint8_t*>(workspace) + p.wpack_off[k];
    const int blocks = pack_grid(s, p.Hp[k], k);
    if (f16) {
      // per-layer max|W_k| -> power-of-two scale, then one fp16 image per chunk
      DTB_CUDA_OK(cudaMemsetAsync(wmax + k, 0, sizeof(int), st));
      const int64_t n_w = (int64_t)s.F * s.H[k] * s.L[k];
      cin_tc_wmax_kernel<<<(int)((n_w + 255) / 256 < 64 ? (n_w + 255) / 256 : 64), 256, 0, st>>>(weights + s.w_off[k], n_w, wmax + k);
      DTB_LAUNCH_OK();
      cin_tc_pack_f16_kernel<<<blocks, 256, 0, st>>>(weights + s.w_off[k], img, s.F, s.H[k], p.Hp[k], s.L[k], wmax + k);
    } else {
      cin_tc_pack_kernel<<<blocks, 256, 0, st>>>(weights + s.w_off[k], img, s.F, s.H[k], p.Hp[k], s.L[k]);
    }
    DTB_LAUNCH_OK();
  }
  if (f16) return cin_tc2_launch_fwd(p, s.D, st);
  const TcSmemLayout lay = tc_layout(bstage, s.F);
#define DTB_TC_LAUNCH(DD) \
  case DD:                \
    return launch_fwd<DD>(p, lay.total, st);
  switch (s.D) {
    DTB_TC_LAUNCH(4)
    DTB_TC_LAUNCH(8)
    DTB_TC_LAUNCH(16)
    DTB_TC_LAUNCH(32)
    default:
      set_error("dtb_cin_fwd: embedding dim %d unsupported by the tensor-core kernel", s.D);
      return DTB_ERR_UNSUPPORTED;
  }
#undef DTB_TC_LAUNCH
}

}  // namespace dtb

using namespace dtb;

extern "C" {

// test hooks (declared in include/deeptables_b200.h)
int dtb_cin_tc_set_variant(int flags) {
  const unsigned unknown = (unsigned)flags & ~(1u | (1u << 16) | (1u << 17));    // bit 0 is accepted and ignored
  if (unknown) {
    set_error("dtb_cin_tc_set_variant: unknown flag bit %d (known: 0, 16, 17)", __builtin_ctz(unknown));
    return DTB_ERR_INVALID_ARG;
  }
  g_tc_bwd_fp32 = (flags >> 16) & 1;  // bit 16: exact-fp32 backward
  g_tc_full_save = (flags >> 17) & 1; // bit 17: full (fp32 T_k) saved activations
  return DTB_OK;
}

int dtb_tc_selftest(const float* A, const float* Bmat, float* C, void* workspace, int N, int K, int a_operand_in_tmem,
                    void* stream) {
  DTB_CHECK_ARG(A && Bmat && C && workspace, "NULL argument");
  DTB_CHECK_ARG(N % 16 == 0 && N >= 16 && N <= 128 && K % 16 == 0 && K >= 16 && K <= 64, "N<=128, K<=64, x16");
  cudaStream_t st = (cudaStream_t)stream;
  // Bmat is [K, N] row-major (a CIN filter with F = 1, H = K): pack -> image (hi | lo)
  cin_tc_pack_kernel<<<32, 256, 0, st>>>(Bmat, reinterpret_cast<uint8_t*>(workspace), 1, K, K, N);
  DTB_LAUNCH_OK();
  const int smem = 2 * 128 * 64 * 2 + 64;
  if (a_operand_in_tmem) {
    DTB_CUDA_OK(cudaFuncSetAttribute(tc_selftest_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    tc_selftest_kernel<true><<<1, 160, smem, st>>>(A, reinterpret_cast<uint8_t*>(workspace), C, N, K);
  } else {
    DTB_CUDA_OK(cudaFuncSetAttribute(tc_selftest_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    tc_selftest_kernel<false><<<1, 160, smem, st>>>(A, reinterpret_cast<uint8_t*>(workspace), C, N, K);
  }
  DTB_LAUNCH_OK();
  return DTB_OK;
}

}  // extern "C"

// ==========================================================================================
// Backward on the tensor cores
// ==========================================================================================
// dgrad (per 2 x 128-row super tile, layers last -> first):
//   dC_k = (d_pooled part + dh_{k+1}) * act'(T_k)            [thread-local: row m = (b,d)]
//   dZ_{k,i}[m, j] = sum_l dC_k[m,l] W_k[(i,j), l]           [UMMA: A = dC (TMEM, written once per layer),
//                                                             B = W_{k,i} K-major in l, N = Hp, K = L]
//   dx0[m,i] += sum_j dZ[m,j] h_k[m,j] ;  dh_k[m,j] += dZ[m,j] x0[m,i]     [epilogue, registers]
//   dC_k is also written to HBM as bf16 hi/lo MN-major tiles for the wgrad kernel.
// wgrad (per layer, grid = i-tile pairs x row splits):
//   dW_k[(i,j), l] = sum_m x0[m,i] h_k[m,j] dC_k[m,l]        [UMMA: A[(i,j), m] built in TMEM from smem tiles
//                                                             of x0t / h_k, B = dC tiles (MN-major, bulk copy)]
namespace dtb {

// weights -> per chunk i: [hi | lo] image of B[n=j][k=l] = W[(i*H + j), l], canonical K-major no swizzle
__global__ void cin_tc_pack_t_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int F, int H, int Hp,
                                     int L) {
  const int64_t per_chunk = (int64_t)L * Hp;
  const int64_t total = per_chunk * F;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(t / per_chunk);
    const int rem = (int)(t - (int64_t)i * per_chunk);
    const int j = rem / L, l = rem - j * L;       // l fastest: coalesced reads
    const float v = j < H ? w[((int64_t)i * H + j) * L + l] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    const int64_t off = ((int64_t)(l >> 3) * (Hp >> 3) + (j >> 3)) * 128 + (j & 7) * 16 + (l & 7) * 2;
    uint8_t* base = out + (int64_t)i * per_chunk * 4;
    *reinterpret_cast<__nv_bfloat16*>(base + off) = hi;
    *reinterpret_cast<__nv_bfloat16*>(base + per_chunk * 2 + off) = lo;
  }
}

// single fp16 pass (cin_tc2.cu): ONE fp16 image per chunk (the "hi" slot) of B[n=j][k=l] = W[(i*H + j), l] * s_W
__global__ void cin_tc_pack_t_f16_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int F, int H, int Hp,
                                         int L, const int* __restrict__ wmax) {
  float s, inv;
  tc::pow2_scale_to_1024(__int_as_float(*wmax), s, inv);
  const int64_t per_chunk = (int64_t)L * Hp;
  const int64_t total = per_chunk * F;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(t / per_chunk);
    const int rem = (int)(t - (int64_t)i * per_chunk);
    const int j = rem / L, l = rem - j * L;       // l fastest: coalesced reads
    const float v = j < H ? w[((int64_t)i * H + j) * L + l] * s : 0.f;
    const int64_t off = ((int64_t)(l >> 3) * (Hp >> 3) + (j >> 3)) * 128 + (j & 7) * 16 + (l & 7) * 2;
    *reinterpret_cast<__half*>(out + (int64_t)i * per_chunk * 4 + off) = __float2half_rn(v);
  }
}

struct TcBwdSmemLayout {
  int b_off, x0_off, dx_off, bar_off, total;
};
__host__ __device__ inline TcBwdSmemLayout tc_bwd_layout(int b_stage_bytes, int F) {
  TcBwdSmemLayout l;
  l.b_off = 0;
  l.x0_off = kStagesB * b_stage_bytes;
  l.dx_off = l.x0_off + 2 * 128 * F * 4;
  l.bar_off = l.dx_off + 2 * 128 * F * 4;
  l.bar_off = (l.bar_off + 15) / 16 * 16;
  l.total = l.bar_off + 256;
  return l;
}

template <int D>
__global__ void __launch_bounds__(kTcThreads, 1) cin_tc_dgrad_kernel(const __grid_constant__ CinTcBwdParams p) {
  constexpr int R = 128 / D;
  extern __shared__ __align__(1024) uint8_t smem[];
  const TcBwdSmemLayout lay = tc_bwd_layout(p.b_stage_bytes, p.F);
  uint8_t* smem_b = smem + lay.b_off;
  float* x0s = reinterpret_cast<float*>(smem + lay.x0_off);
  float* dxs = reinterpret_cast<float*>(smem + lay.dx_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* a_ready = bars;          // [tile]            2
  uint64_t* full_b = bars + 2;       // [stage]           4
  uint64_t* empty_b = bars + 6;      // [stage]           4
  uint64_t* acc_full = bars + 10;    // [tile][buf]       4
  uint64_t* acc_empty = bars + 14;   // [tile][buf]       4
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = p.F;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);

  if (threadIdx.x == 0) {
    tc::mbar_init(&a_ready[0], 4);
    tc::mbar_init(&a_ready[1], 4);
    for (int s = 0; s < kStagesB; ++s) {
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty_b[s], 1);
    }
    for (int i = 0; i < 4; ++i) {
      tc::mbar_init(&acc_full[i], 1);
      tc::mbar_init(&acc_empty[i], 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == 8) tc::tmem_alloc(tmem_slot, kTmemCols);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    const int g = warp >> 2;
    const int t = threadIdx.x & 127;
    const int r = t / D, d = t % D;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t t_tile = tmem_base + lane_base + g * 256;   // A: [0,64) hi [64,128) lo ; acc: 128 + buf*64
    float* x0g = x0s + (size_t)g * 128 * F;    // [r][i][d]
    float* dxg = dxs + (size_t)g * 128 * F;    // [i][t]
    uint32_t acc_cnt = 0;
    float h[kMaxHp], dh[kMaxHp];
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      const int row0 = (st * 2 + g) * R;
      const int b = row0 + r;
      const bool valid = b < p.B;
      const size_t m_pad = (size_t)(st * 2 + g) * 128 + t;    // == b*D + d
      {
        constexpr int Q = D / 4;
        for (int e = t; e < R * F * Q; e += 128) {
          const int rr = e / (F * Q);
          const int rem = e - rr * F * Q;
          const int i = rem / Q, q = rem - i * Q;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row0 + rr < p.B) {
            const int64_t rb = table_row(p.row_offsets, i, __ldg(p.idx + (int64_t)(row0 + rr) * F + i), D, nullptr);
            if (rb >= 0) v = ldg_stream_f4(p.table + rb + (q << 2));
          }
          *reinterpret_cast<float4*>(x0g + ((size_t)rr * F + i) * D + (q << 2)) = v;
        }
        for (int i = 0; i < F; ++i) dxg[i * 128 + t] = 0.f;
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
#pragma unroll
      for (int j = 0; j < kMaxHp; ++j) dh[j] = 0.f;
      for (int k = p.n_layers - 1; k >= 0; --k) {
        const int L = p.L[k], Hp = p.Hp[k];
        const int hid_n = p.hid_n[k], pool_lo = p.pool_lo[k], pool_n = p.pool_n[k];
        // ---- dC_k row -> TMEM A operand (hi|lo) + HBM tiles for wgrad ---------------------------
        const float* Trow = p.saved + p.saved_off[k] + m_pad * L;
        const int mask_words = (L + 31) >> 5;
        uint32_t mw[kMaxL / 32];
#pragma unroll
        for (int w = 0; w < kMaxL / 32; ++w) mw[w] = 0u;
        if (p.compact && p.act == DTB_ACT_RELU && valid) {
          const uint32_t* mrow = reinterpret_cast<const uint32_t*>(p.saved + p.saved_off[k]) + m_pad * mask_words;
#pragma unroll
          for (int w = 0; w < kMaxL / 32; ++w)
            if (w < mask_words) mw[w] = __ldg(mrow + w);
        }
        const float* dprow = p.d_pooled + (size_t)b * p.P + p.pcol0[k];
        uint8_t* dcblk = p.dc_tiles + p.dc_off[k] + (m_pad >> 4) * (size_t)(64 * L) + ((t & 15) >> 3) * 128 + (t & 7) * 16;
#pragma unroll
        for (int cb = 0; cb < kMaxL / 16; ++cb) {
          if (cb * 16 < L) {
            float tv[16];
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              const float4 q4 = (valid && !p.compact) ? *reinterpret_cast<const float4*>(Trow + cb * 16 + j)
                                                      : make_float4(0.f, 0.f, 0.f, 0.f);
              tv[j] = q4.x; tv[j + 1] = q4.y; tv[j + 2] = q4.z; tv[j + 3] = q4.w;
            }
            float dc[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int col = cb * 16 + j;
              float gsum = 0.f;
              if (valid && col >= pool_lo && col < pool_lo + pool_n) gsum = __ldg(dprow + (col - pool_lo));
              if (col < kMaxHp) {
                if (col < hid_n) gsum += dh[col];
              }
              const bool on = p.compact ? (((mw[cb >> 1] >> ((cb & 1) * 16 + j)) & 1u) != 0u) : (tv[j] > 0.f);
              if (p.act == DTB_ACT_RELU && !on) gsum = 0.f;
              dc[j] = valid ? gsum : 0.f;
            }
            uint32_t zh[8], zl[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) tc::split_bf16x2(dc[2 * q], dc[2 * q + 1], zh[q], zl[q]);
            tc::tmem_st8v(t_tile + cb * 8, zh[0], zh[1], zh[2], zh[3], zh[4], zh[5], zh[6], zh[7]);
            tc::tmem_st8v(t_tile + 64 + cb * 8, zl[0], zl[1], zl[2], zl[3], zl[4], zl[5], zl[6], zl[7]);
            *reinterpret_cast<uint4*>(dcblk + (cb * 2) * 256) = make_uint4(zh[0], zh[1], zh[2], zh[3]);
            *reinterpret_cast<uint4*>(dcblk + (cb * 2 + 1) * 256) = make_uint4(zh[4], zh[5], zh[6], zh[7]);
            *reinterpret_cast<uint4*>(dcblk + 32 * L + (cb * 2) * 256) = make_uint4(zl[0], zl[1], zl[2], zl[3]);
            *reinterpret_cast<uint4*>(dcblk + 32 * L + (cb * 2 + 1) * 256) = make_uint4(zl[4], zl[5], zl[6], zl[7]);
            tc::tmem_wait_st();
          }
        }
        tc::fence_before_thread_sync();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&a_ready[g]);
        // ---- h_k (this row's slice) and a fresh dh accumulator ------------------------------------
        if (k > 0) {
          const int Hk = p.H[k];
          if (p.compact) {
            // [m / 64][j][68] tiles written by the forward for wgrad: for a fixed j the 64 rows of a block are contiguous
            const float* hbp = p.saved + p.hb_off[k - 1] + (m_pad >> 6) * (size_t)(Hk * kWgPad) + (m_pad & 63);
#pragma unroll
            for (int j = 0; j < kMaxHp; ++j) h[j] = (valid && j < Hk) ? __ldg(hbp + (size_t)j * kWgPad) : 0.f;
          } else {
            const float* prow = p.saved + p.saved_off[k - 1] + m_pad * p.L[k - 1];
#pragma unroll
            for (int j = 0; j < kMaxHp; j += 4) {
              float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f);
              if (valid && j < Hk) q4 = *reinterpret_cast<const float4*>(prow + j);   // H_k is a multiple of 4 (L/2, L % 16 == 0)
              h[j] = q4.x; h[j + 1] = q4.y; h[j + 2] = q4.z; h[j + 3] = q4.w;
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < kMaxHp; ++j) h[j] = (j < F) ? x0g[((size_t)r * F + j) * D + d] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < kMaxHp; ++j) dh[j] = 0.f;
        for (int i = 0; i < F; ++i) {
          const uint32_t buf = acc_cnt & 1, par = (acc_cnt >> 1) & 1;
          ++acc_cnt;
          const float xi = x0g[((size_t)r * F + i) * D + d];
          tc::mbar_wait(&acc_full[g * 2 + buf], par);
          tc::fence_after_thread_sync();
          float dx = 0.f;
#pragma unroll
          for (int cb = 0; cb < kMaxHp / 16; ++cb) {
            if (cb * 16 < Hp) {
              uint32_t v[16];
              tc::tmem_ld16(t_tile + 128 + buf * 64 + cb * 16, v);
              tc::tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float dz = __uint_as_float(v[j]);
                dx = fmaf(dz, h[cb * 16 + j], dx);
                dh[cb * 16 + j] = fmaf(dz, xi, dh[cb * 16 + j]);
              }
            }
          }
          tc::fence_before_thread_sync();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&acc_empty[g * 2 + buf]);
          dxg[i * 128 + t] += dx;
        }
        if (k == 0) {
#pragma unroll
          for (int j = 0; j < kMaxHp; ++j)
            if (j < F) dxg[j * 128 + t] += dh[j];     // h_0 is x0 itself
        }
      }
      // ---- scatter dx0 of this tile into the embedding gradient ------------------------------------
      if (valid) {
        for (int i = 0; i < F; ++i) {
          const int64_t rb = table_row(p.row_offsets, i, __ldg(p.idx + (int64_t)b * F + i), D, nullptr);
          if (rb >= 0) atomicAdd(p.grad_table + rb + d, dxg[i * 128 + t]);
        }
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
    }
  } else if (warp == 8) {
    const bool leader = elect_one_sync();
    const uint32_t smem_b_u32 = tc::smem_u32(smem_b);
    uint32_t chunk = 0, cnt0 = 0, cnt1 = 0, layer_cnt = 0;
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      for (int k = p.n_layers - 1; k >= 0; --k, ++layer_cnt) {
        const int Hp = p.Hp[k], L = p.L[k];
        const uint32_t idesc = tc::make_idesc_bf16(128, (uint32_t)Hp);
        const uint32_t lbo_b = (uint32_t)(Hp >> 3) * 128;
        const uint32_t img_b = (uint32_t)L * Hp * 2;
        const uint64_t desc_hi = ((uint64_t)((lbo_b >> 4) & 0x3FFF) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
        for (int i = 0; i < F; ++i, ++chunk) {
          const uint32_t sb = chunk % kStagesB, pb = (chunk / kStagesB) & 1;
          tc::mbar_wait(&full_b[sb], pb);
          const uint32_t b_addr = smem_b_u32 + sb * (uint32_t)p.b_stage_bytes;
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            if (i == 0) tc::mbar_wait(&a_ready[g], layer_cnt & 1);
            const uint32_t c = g ? cnt1 : cnt0;
            const uint32_t buf = c & 1, par = (c >> 1) & 1;
            if (g) ++cnt1; else ++cnt0;
            tc::mbar_wait(&acc_empty[g * 2 + buf], par ^ 1);
            tc::fence_after_thread_sync();
            if (leader) {
              const uint32_t a_base = tmem_base + g * 256;
              const uint32_t d_tmem = a_base + 128 + buf * 64;
#pragma unroll
              for (int pass = 0; pass < 3; ++pass) {
                if (pass < p.n_pass) {
                  const uint32_t a_addr = a_base + (pass == 1 ? 64 : 0);
                  const uint32_t b_img = b_addr + (pass == 2 ? img_b : 0);
#pragma unroll
                  for (int ks = 0; ks < kMaxL / 16; ++ks) {
                    if (ks * 16 < L) {
                      const uint64_t desc_b = desc_hi | (uint64_t)(((b_img + ks * 2 * lbo_b) >> 4) & 0x3FFF);
                      tc::mma_ts(d_tmem, a_addr + ks * 8, desc_b, idesc, (uint32_t)((pass | ks) != 0));
                    }
                  }
                }
              }
              tc::mma_commit(&acc_full[g * 2 + buf]);
            }
            __syncwarp();
          }
          if (leader) tc::mma_commit(&empty_b[sb]);
          __syncwarp();
        }
      }
    }
  } else {
    if (lane == 0) {
      uint32_t chunk = 0;
      for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
        for (int k = p.n_layers - 1; k >= 0; --k) {
          const uint32_t bytes = (uint32_t)p.L[k] * p.Hp[k] * 2 * (p.n_pass > 1 ? 2 : 1);
          const uint32_t stride = (uint32_t)p.L[k] * p.Hp[k] * 4;
          const uint8_t* src = p.wpack + p.wpack_off[k];
          for (int i = 0; i < F; ++i, ++chunk) {
            const uint32_t sb = chunk % kStagesB, pb = (chunk / kStagesB) & 1;
            tc::mbar_wait(&empty_b[sb], pb ^ 1);
            tc::mbar_arrive_expect_tx(&full_b[sb], bytes);
            tc::bulk_g2s(smem_b + (size_t)sb * p.b_stage_bytes, src + (size_t)i * stride, bytes, &full_b[sb]);
          }
        }
      }
    }
    __syncwarp();
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 8) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}


// ------------------------------------------------------------------------------------------
// wgrad kernel (one launch per layer)
// ------------------------------------------------------------------------------------------
constexpr int kWgThreads = 384;     // warps 0-3 / 4-7: A producers of tile 0 / 1 (+ final epilogue), 8: MMA, 9: dC bulk loader,
                                    // 10-11: h / x0 tile loaders
constexpr int kWgStageRows = 64;    // GEMM-K (batch x dim rows) per pipeline stage = 4 UMMA k-steps
constexpr int kWgStages = 3;
constexpr int kWgStagesA = 2;

struct CinTcWgradParams {
  const float* xb;           // block-transposed x0:  [M_pad/64][F][68]
  const float* hb;           // block-transposed h_k: [M_pad/64][H][68]  (== xb for layer 0)
  const uint8_t* dc_tiles;   // layer k blocks of 16 rows: [hi 32*L B | lo 32*L B]
  float* d_w;                // [F*H, L] accumulate
  int F, H, Hp, L, n_pass;
  int n_stage_total;         // ceil(M_pad / 64)
  int stages_per_split;
};

struct WgSmemLayout {
  int b_off, h_off, x_off, bar_off, total, b_bytes, h_bytes, x_bytes;
};
__host__ __device__ inline WgSmemLayout wg_layout(int L, int Hp, int F) {
  WgSmemLayout l;
  l.b_bytes = 4 * 64 * L;                       // 4 blocks of 16 rows, hi + lo
  l.h_bytes = Hp * kWgPad * 4;
  l.x_bytes = F * kWgPad * 4;
  l.b_off = 0;
  l.h_off = kWgStages * l.b_bytes;
  l.x_off = l.h_off + kWgStages * l.h_bytes;
  l.bar_off = l.x_off + kWgStages * l.x_bytes;
  l.total = l.bar_off + 256;
  return l;
}

__global__ void __launch_bounds__(kWgThreads, 1) cin_tc_wgrad_kernel(const __grid_constant__ CinTcWgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const WgSmemLayout lay = wg_layout(p.L, p.Hp, p.F);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* full_b = bars;            // [stage] 3   dC tiles landed (tx)
  uint64_t* empty_b = bars + 3;       // [stage] 3   MMA done with the dC tiles
  uint64_t* full_h = bars + 6;        // [stage] 3   h / x0 tiles written (2 loader warps)
  uint64_t* empty_h = bars + 9;       // [stage] 3   all 8 producer warps done reading them
  uint64_t* full_a = bars + 12;       // [tile][stageA] 4
  uint64_t* empty_a = bars + 16;      // [stageA] 2
  uint64_t* acc_done = bars + 18;     // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = p.F, H = p.H, Hp = p.Hp, L = p.L;
  const int ipt = 128 / Hp;                              // x0 fields per 128-row tile
  const int s_begin = blockIdx.y * p.stages_per_split;
  int s_end = s_begin + p.stages_per_split;
  if (s_end > p.n_stage_total) s_end = p.n_stage_total;
  const int n_st = s_end > s_begin ? s_end - s_begin : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kWgStages; ++s) {
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty_b[s], 1);
      tc::mbar_init(&full_h[s], 1);
      tc::mbar_init(&empty_h[s], 8);
    }
    for (int i = 0; i < 4; ++i) tc::mbar_init(&full_a[i], 4);
    tc::mbar_init(&empty_a[0], 1);
    tc::mbar_init(&empty_a[1], 1);
    tc::mbar_init(acc_done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 8) tc::tmem_alloc(tmem_slot, kTmemCols);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // ---- A producers: lane row = (il, j): A[row, m] = x0[m, i] * h[m, j] ---------------------------
    const int g = warp >> 2;
    const int t = threadIdx.x & 127;
    const int il = t / Hp, j = t - il * Hp;
    const int i = (blockIdx.x * 2 + g) * ipt + il;
    const bool live = (i < F) && (j < H);
    const bool h_is_x = (p.hb == p.xb);
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    for (int s = 0; s < n_st; ++s) {
      const uint32_t sh = s % kWgStages, ph = (s / kWgStages) & 1;
      const uint32_t sa = s % kWgStagesA, pa = (s / kWgStagesA) & 1;
      const float* xs = reinterpret_cast<const float*>(smem + lay.x_off + sh * lay.x_bytes);
      const float* hs = h_is_x ? xs : reinterpret_cast<const float*>(smem + lay.h_off + sh * lay.h_bytes);
      tc::mbar_wait(&full_h[sh], ph);
      // this lane's x0 field row and hidden-field row of the stage, 64 consecutive batch*dim rows each
      const float4* xrow = reinterpret_cast<const float4*>(xs + (live ? i : 0) * kWgPad);
      const float4* hrow = reinterpret_cast<const float4*>(hs + (live ? j : 0) * kWgPad);
      uint32_t zh[32], zl[32];
#pragma unroll
      for (int q4 = 0; q4 < 16; ++q4) {
        const float4 xv = xrow[q4], hv = hrow[q4];
        const float sc = live ? 1.f : 0.f;
        tc::split_bf16x2(xv.x * hv.x * sc, xv.y * hv.y * sc, zh[2 * q4], zl[2 * q4]);
        tc::split_bf16x2(xv.z * hv.z * sc, xv.w * hv.w * sc, zh[2 * q4 + 1], zl[2 * q4 + 1]);
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&empty_h[sh]);
      tc::mbar_wait(&empty_a[sa], pa ^ 1);
      tc::fence_after_thread_sync();
      const uint32_t a_col = tmem_base + lane_base + 256 + (sa * 2 + g) * 64;   // per k-step: 8 hi + 8 lo columns
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        tc::tmem_st8v(a_col + ks * 16, zh[ks * 8 + 0], zh[ks * 8 + 1], zh[ks * 8 + 2], zh[ks * 8 + 3], zh[ks * 8 + 4],
                      zh[ks * 8 + 5], zh[ks * 8 + 6], zh[ks * 8 + 7]);
        tc::tmem_st8v(a_col + ks * 16 + 8, zl[ks * 8 + 0], zl[ks * 8 + 1], zl[ks * 8 + 2], zl[ks * 8 + 3], zl[ks * 8 + 4],
                        zl[ks * 8 + 5], zl[ks * 8 + 6], zl[ks * 8 + 7]);
      }
      tc::tmem_wait_st();
      tc::fence_before_thread_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&full_a[g * kWgStagesA + sa]);
    }
    // ---- epilogue: accumulator row -> dW[(i,j), :] ---------------------------------------------------
    if (n_st > 0) {
      tc::mbar_wait(acc_done, 0);
      tc::fence_after_thread_sync();
      float* dst = p.d_w + ((size_t)i * H + j) * L;
#pragma unroll
      for (int cb = 0; cb < kMaxL / 16; ++cb) {
        if (cb * 16 < L) {
          uint32_t v[16];
          tc::tmem_ld16(tmem_base + lane_base + g * kAccCols + cb * 16, v);
          tc::tmem_wait_ld();
          if (live) {
#pragma unroll
            for (int q = 0; q < 16; ++q) atomicAdd(dst + cb * 16 + q, __uint_as_float(v[q]));
          }
        }
      }
      tc::fence_before_thread_sync();
    }
  } else if (warp == 8) {
    const bool leader = elect_one_sync();
    const uint32_t idesc = tc::make_idesc_bf16_bmn(128, (uint32_t)L);
    // dC tile descriptor (MN-major): LBO = 128 B (k-group), SBO = 256 B (n-group)
    const uint64_t desc_hi = ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
    const uint32_t smem_b_u32 = tc::smem_u32(smem + lay.b_off);
    for (int s = 0; s < n_st; ++s) {
      const uint32_t sb = s % kWgStages, pb = (s / kWgStages) & 1;
      const uint32_t sa = s % kWgStagesA, pa = (s / kWgStagesA) & 1;
      tc::mbar_wait(&full_b[sb], pb);
      const uint32_t b_addr = smem_b_u32 + sb * (uint32_t)lay.b_bytes;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        tc::mbar_wait(&full_a[g * kWgStagesA + sa], pa);
        tc::fence_after_thread_sync();
        if (leader) {
          const uint32_t d_tmem = tmem_base + g * kAccCols;
          const uint32_t a_base = tmem_base + 256 + (sa * 2 + g) * 64;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
              if (pass < p.n_pass) {
                // pass 0: Z_hi*dC_hi ; 1: Z_lo*dC_hi ; 2: Z_hi*dC_lo
                const uint32_t a_addr = a_base + ks * 16 + (pass == 1 ? 8 : 0);
                const uint32_t blk = b_addr + ks * (64 * L) + (pass == 2 ? 32 * L : 0);
                const uint64_t desc_b = desc_hi | (uint64_t)((blk >> 4) & 0x3FFF);
                tc::mma_ts(d_tmem, a_addr, desc_b, idesc, (uint32_t)((s | ks | pass) != 0));
              }
            }
          }
        }
        __syncwarp();
      }
      if (leader) {
        tc::mma_commit(&empty_a[sa]);
        tc::mma_commit(&empty_b[sb]);
        if (s == n_st - 1) tc::mma_commit(acc_done);
      }
      __syncwarp();
    }
  } else if (warp == 9) {
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)lay.b_bytes;
      for (int s = 0; s < n_st; ++s) {
        const uint32_t sb = s % kWgStages, pb = (s / kWgStages) & 1;
        tc::mbar_wait(&empty_b[sb], pb ^ 1);
        tc::mbar_arrive_expect_tx(&full_b[sb], bytes);
        tc::bulk_g2s(smem + lay.b_off + sb * lay.b_bytes, p.dc_tiles + (size_t)(s_begin + s) * bytes, bytes, &full_b[sb]);
      }
    }
    __syncwarp();
  } else {
    // ---- x0 / h tile loader (warp 10): one bulk async copy each per 64-row stage ------------------
    if (warp == 10 && lane == 0) {
      const bool h_is_x = (p.hb == p.xb);
      const uint32_t x_bytes = (uint32_t)lay.x_bytes, h_bytes = (uint32_t)(H * kWgPad * 4);
      for (int s = 0; s < n_st; ++s) {
        const uint32_t sh = s % kWgStages, ph = (s / kWgStages) & 1;
        tc::mbar_wait(&empty_h[sh], ph ^ 1);
        const size_t blk = (size_t)(s_begin + s);
        tc::mbar_arrive_expect_tx(&full_h[sh], x_bytes + (h_is_x ? 0u : h_bytes));
        tc::bulk_g2s(smem + lay.x_off + sh * lay.x_bytes, p.xb + blk * (size_t)(F * kWgPad), x_bytes, &full_h[sh]);
        if (!h_is_x)
          tc::bulk_g2s(smem + lay.h_off + sh * lay.h_bytes, p.hb + blk * (size_t)(H * kWgPad), h_bytes, &full_h[sh]);
      }
    }
    __syncwarp();
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 8) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// d_bias[l] += sum over rows of dC (hi + lo of the tiles): only when the CIN has biases
__global__ void cin_tc_dbias_kernel(const uint8_t* __restrict__ dc_tiles, float* __restrict__ d_bias, int L,
                                    int n_blocks16) {
  // thread per (block of 16 rows, l); tile layout: [n_grp][k_grp 2][8 rows][8 l]
  const int64_t total = (int64_t)n_blocks16 * L;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t blk = t / L;
    const int l = (int)(t - blk * L);
    const uint8_t* base = dc_tiles + blk * (int64_t)(64 * L) + (l >> 3) * 256 + (l & 7) * 2;
    float s = 0.f;
    for (int hl = 0; hl < 2; ++hl)
      for (int m = 0; m < 16; ++m)
        s += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(base + hl * 32 * L + (m >> 3) * 128 + (m & 7) * 16));
    if (s != 0.f) atomicAdd(d_bias + l, s);
  }
}

// ------------------------------------------------------------------------------------------
// host side of the backward
// ------------------------------------------------------------------------------------------
static size_t dc_bytes(const CinShape& s, int B, size_t* off /* per layer */) {
  const int R = 128 / s.D;
  const size_t n_super = ((size_t)B + 2 * R - 1) / (2 * R);
  const size_t m_pad = n_super * 256;
  size_t total = 0;
  for (int k = 0; k < s.n_layers; ++k) {
    if (off) off[k] = total;
    total += (m_pad / 16) * (size_t)(64 * s.L[k]);
  }
  return total;
}

// [packed weights | dC tiles | 1024 B slack whose last 256 B are the statistics words | cin_tc2: max|d_pooled| per
// (batch row, layer) + 64 B of shape tables]
static size_t bwd_stats_end(const CinShape& s, int B) { return wpack_bytes(s) + 1024 + dc_bytes(s, B, nullptr) + 1024; }
size_t cin_tc_bwd_workspace_bytes(const CinShape& s, int B) {
  return bwd_stats_end(s, B) + (size_t)B * kCinMaxLayers * sizeof(float) + 256;
}

template <int D>
static int launch_dgrad(const CinTcBwdParams& p, int smem_bytes, cudaStream_t st) {
  auto kern = cin_tc_dgrad_kernel<D>;
  DTB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  const int R = 128 / D;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);
  int grid = sm_count();
  if (grid > n_super) grid = n_super;
  kern<<<grid, kTcThreads, smem_bytes, st>>>(p);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

static bool cin_tc_bwd_supported(const CinShape& s) {
  if (!cin_tc_supported(s)) return false;
  int bstage = 0;
  for (int k = 0; k < s.n_layers; ++k) {
    const int bytes = 4 * s.L[k] * round_up(s.H[k], kSubK);
    if (bytes > bstage) bstage = bytes;
    if (s.H[k] % 4 && k > 0) return false;
    if (wg_layout(s.L[k], round_up(s.H[k], kSubK), s.F).total > 227 * 1024) return false;
  }
  return tc_bwd_layout(bstage, s.F).total <= 227 * 1024;
}

int cin_tc_bwd(const CinShape& s, const int32_t* idx, const float* table, const int64_t* row_offsets,
               const float* weights, const float* d_pooled, const void* saved, float* grad_table,
               float* d_weights, float* d_bias, void* workspace, size_t workspace_bytes, int B, int act,
               int n_pass, int f16, int phase, cudaStream_t st) {
  // phase 0: everything; 1: the embedding-gradient part (weight pack + dgrad); 2: the weight-gradient part
  // (wgrad + bias).  Lets the host start the data-parallel exchange of the table gradient under the wgrad.
  if (!cin_tc_bwd_supported(s) || g_tc_bwd_fp32) {
    if (phase == 2) return DTB_OK;
    return cin_fp32_bwd(s, idx, table, row_offsets, weights, d_pooled, saved, grad_table, d_weights, d_bias,
                        workspace, workspace_bytes, B, act, st);
  }
  if (workspace_bytes < cin_tc_bwd_workspace_bytes(s, B)) {
    set_error("dtb_cin_bwd: workspace too small for the tensor-core backward");
    return DTB_ERR_INVALID_ARG;
  }
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  const size_t wp = (wpack_bytes(s) + 1023) / 1024 * 1024;
  CinTcBwdParams p{};
  p.idx = idx; p.table = table; p.row_offsets = row_offsets;
  p.wpack = ws; p.d_pooled = d_pooled; p.saved = reinterpret_cast<const float*>(saved);
  p.grad_table = grad_table; p.dc_tiles = ws + wp;
  p.B = B; p.F = s.F; p.n_layers = s.n_layers; p.act = act; p.n_pass = n_pass; p.P = s.P;
  size_t dc_off[kCinMaxLayers];
  dc_bytes(s, B, dc_off);
  size_t woff = 0, soff = (size_t)B * s.D * s.F;
  p.compact = cin_tc_compact(s) ? 1 : 0;
  const size_t bt_blocks = m_pad_rows(s, B) / 64;
  const size_t xb_pos = cin_fp32_saved_bytes(s, B) / sizeof(float);      // block-transposed tiles, as cin_tc_fwd
  size_t hoff = xb_pos + bt_blocks * s.F * kWgPad;
  int bstage = 0;
  for (int k = 0; k < s.n_layers; ++k) {
    p.L[k] = s.L[k]; p.H[k] = s.H[k]; p.Hp[k] = round_up(s.H[k], kSubK);
    p.pool_lo[k] = s.pool_lo[k]; p.pool_n[k] = s.pool_n[k]; p.pcol0[k] = s.pcol0[k];
    p.hid_n[k] = (k + 1 < s.n_layers) ? s.H[k + 1] : 0;
    p.wpack_off[k] = woff; p.saved_off[k] = soff; p.dc_off[k] = dc_off[k];
    p.hb_off[k] = hoff;
    hoff += bt_blocks * p.hid_n[k] * kWgPad;
    const size_t chunk = (size_t)s.L[k] * p.Hp[k] * 4;
    woff += chunk * s.F;
    soff += (size_t)B * s.D * s.L[k];
    if ((int)chunk > bstage) bstage = (int)chunk;
  }
  p.b_stage_bytes = bstage;
  // statistics words of the single fp16 pass, read by the cin_tc2.cu kernels: [k] max|W_k|, [8 + k] max|dC_k|,
  // [16] max|x0|, [24 + k] max|h_k| (bit patterns of non-negative floats)
  int* stats = reinterpret_cast<int*>(ws + bwd_stats_end(s, B) - 256);
  if (f16) {
    // the two-threads-per-row data-gradient kernel of cin_tc2.cu, whose fp16 dC tiles its weight-gradient kernel reads
    if (!cin_tc2_bwd_supported(p, s.D)) {
      set_error("dtb_cin_bwd: fp16 single pass: shape outside cin_tc2 (F=%d D=%d); use precision 0/2", s.F, s.D);
      return DTB_ERR_UNSUPPORTED;
    }
    float* dpmax = reinterpret_cast<float*>(ws + bwd_stats_end(s, B));
    p.wmax = stats;
    p.dpmax = dpmax;
    if (phase != 2) {
      const int rcd = cin_tc2_dpmax(d_pooled, dpmax, s.pcol0, s.pool_n, B, s.P, s.n_layers, st);
      if (rcd != DTB_OK) return rcd;
      DTB_CUDA_OK(cudaMemsetAsync(stats, 0, 256, st));
      for (int k = 0; k < s.n_layers; ++k) {
        const int64_t n_w = (int64_t)s.F * s.H[k] * s.L[k];
        cin_tc_wmax_kernel<<<(int)((n_w + 255) / 256 < 64 ? (n_w + 255) / 256 : 64), 256, 0, st>>>(weights + s.w_off[k], n_w, stats + k);
        DTB_LAUNCH_OK();
        cin_tc_pack_t_f16_kernel<<<pack_grid(s, p.Hp[k], k), 256, 0, st>>>(weights + s.w_off[k], ws + p.wpack_off[k], s.F, s.H[k], p.Hp[k],
                                                                 s.L[k], stats + k);
        DTB_LAUNCH_OK();
      }
      // operand maxima recorded by cin_tc2_fwd_kernel at the head of the saved buffer -> statistics words of the wgrad
      const int* sv = reinterpret_cast<const int*>(saved);
      DTB_CUDA_OK(cudaMemcpyAsync(stats + 16, sv, sizeof(int), cudaMemcpyDeviceToDevice, st));
      DTB_CUDA_OK(cudaMemcpyAsync(stats + 24, sv, sizeof(int) * s.n_layers, cudaMemcpyDeviceToDevice, st));
      const int rc = cin_tc2_launch_dgrad(p, s.D, st);
      if (rc != DTB_OK) return rc;
    }
  } else if (phase != 2) {
    for (int k = 0; k < s.n_layers; ++k) {
      cin_tc_pack_t_kernel<<<pack_grid(s, p.Hp[k], k), 256, 0, st>>>(weights + s.w_off[k], ws + p.wpack_off[k], s.F, s.H[k], p.Hp[k], s.L[k]);
      DTB_LAUNCH_OK();
    }
    const int smem = tc_bwd_layout(bstage, s.F).total;
    int rc = DTB_OK;
    switch (s.D) {
      case 4: rc = launch_dgrad<4>(p, smem, st); break;
      case 8: rc = launch_dgrad<8>(p, smem, st); break;
      case 16: rc = launch_dgrad<16>(p, smem, st); break;
      case 32: rc = launch_dgrad<32>(p, smem, st); break;
      default: set_error("dtb_cin_bwd: embedding dim %d unsupported", s.D); return DTB_ERR_UNSUPPORTED;
    }
    if (rc != DTB_OK) return rc;
  }
  if (phase == 1) return DTB_OK;
  // ---- wgrad, one launch per layer ------------------------------------------------------------
  const size_t m_pad = m_pad_rows(s, B);
  const float* xb = reinterpret_cast<const float*>(saved) + xb_pos;
  const float* hb = xb + bt_blocks * s.F * kWgPad;
  for (int k = 0; k < s.n_layers; ++k) {
    const float* hk = k == 0 ? xb : hb;       // block-transposed copies written by the forward kernel
    if (k > 0) hb += bt_blocks * s.H[k] * kWgPad;
    const uint8_t* dc = p.dc_tiles + dc_off[k];
    float* d_w = d_weights + s.w_off[k];
    const int n_stage_total = (int)(m_pad / kWgStageRows);
    if (f16) {
      const int rcw = cin_tc2_launch_wgrad(xb, hk, dc, d_w, s.F, s.H[k], p.Hp[k], s.L[k], n_stage_total, stats, k, st);
      if (rcw != DTB_OK) return rcw;
      if (d_bias) {
        const int rcb = cin_tc2_dbias(dc, d_bias + s.b_off[k], s.L[k], (int)(m_pad / 16), st);
        if (rcb != DTB_OK) return rcb;
      }
      continue;
    }
    CinTcWgradParams w{};
    w.xb = xb; w.hb = hk; w.dc_tiles = dc; w.d_w = d_w;
    w.F = s.F; w.H = s.H[k]; w.Hp = p.Hp[k]; w.L = s.L[k]; w.n_pass = n_pass;
    w.n_stage_total = n_stage_total;
    const int ipt = 128 / w.Hp;
    const int n_tiles = (s.F + ipt - 1) / ipt;
    const int n_pairs = (n_tiles + 1) / 2;
    int splits = sm_count() / n_pairs;
    if (splits < 1) splits = 1;
    if (splits > w.n_stage_total) splits = w.n_stage_total;
    w.stages_per_split = (w.n_stage_total + splits - 1) / splits;
    splits = (w.n_stage_total + w.stages_per_split - 1) / w.stages_per_split;
    const WgSmemLayout wl = wg_layout(w.L, w.Hp, w.F);
    DTB_CUDA_OK(cudaFuncSetAttribute(cin_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wl.total));
    cin_tc_wgrad_kernel<<<dim3(n_pairs, splits), kWgThreads, wl.total, st>>>(w);
    DTB_LAUNCH_OK();
    if (d_bias) {
      const int n_blocks16 = (int)(m_pad / 16);
      int blocks = (int)(((int64_t)n_blocks16 * w.L + 255) / 256);
      if (blocks > sm_count() * 8) blocks = sm_count() * 8;
      cin_tc_dbias_kernel<<<blocks, 256, 0, st>>>(dc, d_bias + s.b_off[k], w.L, n_blocks16);
      DTB_LAUNCH_OK();
    }
  }
  return DTB_OK;
}

}  // namespace dtb
