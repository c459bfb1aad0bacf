// CIN on tcgen05, second organisation: ONE tensor pass on power-of-two-scaled fp16 operands (DTB_CIN_TC_F16X1) with
// TWO threads per GEMM row.
//
// Why a second organisation.  With a single tensor pass the MMA work of a one-thread-per-row fp16 forward built like
// cin_tc_fwd_kernel<D> (cin_tc.cu; removed, it remains in git history at commit 021caee) dropped to a third, but its
// time only fell from 2.54 to 1.90 ms (B200, 65 536 rows): the kernel was never waiting for the tensor pipe any
// more, it was waiting for ITSELF -- 130 pipeline granules per super tile, each a serial chain
// (products -> wait empty -> tcgen05.st -> wait::st -> arrive -> MMA issuer: wait tile 0, issue, wait tile 1, issue, 2 commits)
// of roughly a thousand cycles for 256 cycles of tensor work.  Here:
//   * a granule is one x0 field x ALL hidden fields (K = Hp, up to 64): 78 granules per super tile instead of 130, and
//     twice the tensor work behind every handshake;
//   * both M = 128 tiles of the CTA share one "operand ready" barrier per stage (16 warp arrivals): the issuing warp
//     waits once per granule, issues 2 x Hp/16 MMAs, commits twice;
//   * each GEMM row m = (batch row, dim) is owned by a PAIR of threads, each holding half of h_k[b, :, d] in registers
//     (32 values instead of 64): 16 producer warps instead of 8 hide the tcgen05.st / mbarrier latencies of one
//     another, each writes half of the operand columns, and the accumulator read-out of a layer is split between the
//     two (halves the epilogue, which nothing overlaps because the next layer's operand depends on it);
//   * the fp16 operand of a granule is 32 TMEM columns per tile: 4 stages x 2 tiles = 256 columns next to the two
//     128-column accumulators (TMEM 100 % allocated, as before).
// Arithmetic: per-row scale 2^e chosen from max|x0 row| * max|h row| (the two halves exchange their maxima through
// shared memory), per-layer weight scale from max|W_k|, both undone on the fp32 accumulator.
#include "cin_tc_common.cuh"
#include <cuda_fp16.h>

namespace dtb {

constexpr int kT2Threads = 640;        // warps 0-15 producer + epilogue, 16 / 17 MMA issue for tile 0 / 1 (16 owns TMEM), 18 / 19 weight loaders
constexpr int kT2StagesA = 4;
constexpr int kT2StagesB = 4;          // weight stages PER TILE (forward: each tile streams its own copy of the chunks)
constexpr int kT2ACols = 32;           // TMEM columns of one (stage, tile) operand block: fp16 [128 x 64]

struct T2Smem {
  int b_off, x0_off, mx_off, bar_off, total;
};
__host__ __device__ inline T2Smem tc2_layout(int b_stage_bytes, int F) {
  T2Smem l;
  l.b_off = 0;
  l.x0_off = 2 * kT2StagesB * b_stage_bytes;      // one weight ring per tile
  l.mx_off = l.x0_off + 2 * 128 * F * 4;          // x0s[tile][r][i][d]
  l.bar_off = l.mx_off + 2 * 2 * 2 * 128 * 4;     // row maxima [tile][parity][half][t]
  l.bar_off = (l.bar_off + 15) / 16 * 16;
  l.total = l.bar_off + 320;
  return l;
}

template <int D>
__global__ void __launch_bounds__(kT2Threads, 1) cin_tc2_fwd_kernel(const __grid_constant__ CinTcParams p) {
  constexpr int R = 128 / D;                 // batch rows per M=128 tile
  extern __shared__ __align__(1024) uint8_t smem[];
  const T2Smem lay = tc2_layout(p.b_stage_bytes, p.F);
  uint8_t* smem_b = smem + lay.b_off;
  float* x0s = reinterpret_cast<float*>(smem + lay.x0_off);
  float* mxs = reinterpret_cast<float*>(smem + lay.mx_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  // The two M = 128 tiles of the CTA run INDEPENDENT pipelines (own operand stages, own weight ring, own issuing warp
  // and loader) and tile 1 starts half a layer late: while one tile reads out its accumulator -- which nothing of its own
  // can overlap, the next layer's operand depends on it -- the other tile's MMAs keep the tensor pipe busy.  Sharing each
  // weight chunk between the tiles, as the bf16x3 kernel does, would lock them in step; with ONE fp16 image per chunk
  // two private streams cost what its shared hi + lo stream costs (~21 B/clk/SM from L2).
  uint64_t* full_a = bars;                        // [tile][stage] 8 producer warps
  uint64_t* empty_a = bars + 8;                   // [tile][stage] commit
  uint64_t* full_b = bars + 16;                   // [tile][stage] bulk copy (tx)
  uint64_t* empty_b = bars + 24;                  // [tile][stage] commit
  uint64_t* acc_full = bars + 32;                 // [tile] commit after the last granule of a layer
  uint64_t* start1 = bars + 34;                   // tile 0's issuer -> tile 1: go (after half of tile 0's first layer)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = p.F;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2 * kT2StagesA; ++s) {
      tc::mbar_init(&full_a[s], 8);
      tc::mbar_init(&empty_a[s], 1);
    }
    for (int s = 0; s < 2 * kT2StagesB; ++s) {
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty_b[s], 1);
    }
    tc::mbar_init(&acc_full[0], 1);
    tc::mbar_init(&acc_full[1], 1);
    tc::mbar_init(start1, 1);
    tc::fence_barrier_init();
  }
  if (warp == 16) tc::tmem_alloc(tmem_slot, kTmemCols);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 16) {
    // =================== producer + epilogue: tile g, half q of GEMM row t ============================
    const int g = warp >> 3, q = (warp >> 2) & 1;
    const int t = (warp & 3) * 32 + lane;
    const int tt = q * 128 + t;                     // index inside the tile's 256-thread group
    const int r = t / D, d = t % D;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    float* x0g = x0s + (size_t)g * 128 * F;         // [r][i][d]
    float* mxg = mxs + (size_t)g * 2 * 2 * 128;     // [parity][half][t]
    uint32_t gran = 0, layer_cnt = 0;
    float h[32];
    if (g == 1) tc::mbar_wait(start1, 0);           // stagger: see the barrier table above
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      const int row0 = (st * 2 + g) * R;
      const int b = row0 + r;
      // ---- gather this tile's x0 block: R rows x F fields x D floats, 16-byte pieces, 256 threads ------------
      {
        constexpr int Q = D / 4;
        for (int e = tt; e < R * F * Q; e += 256) {
          const int rr = e / (F * Q);
          const int rem = e - rr * F * Q;
          const int i = rem / Q, qq = rem - i * Q;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row0 + rr < p.B) {
            const int64_t rb = table_row(p.row_offsets, i, __ldg(p.idx + (int64_t)(row0 + rr) * F + i), D, p.status);
            if (rb >= 0) v = ldg_stream_f4(p.table + rb + (qq << 2));
          }
          *reinterpret_cast<float4*>(x0g + ((size_t)rr * F + i) * D + (qq << 2)) = v;
        }
      }
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
      // ---- h_0 = this thread's half of the x0 row (zero padded to Hp[0]) ; max|x0 row| --------------------------
      {
        const int nh0 = p.Hp[0] >> 1;
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) {
          const int j = q * nh0 + jj;
          h[jj] = (jj < nh0 && j < F) ? x0g[((size_t)r * F + j) * D + d] : 0.f;
        }
      }
      float xmax = 0.f;
      for (int i = 0; i < F; ++i) xmax = fmaxf(xmax, fabsf(x0g[((size_t)r * F + i) * D + d]));
      float hmax = xmax;                               // max|h_k row| over BOTH halves
      if (p.saved && q == 0) {
        // maxima of the operand tiles for the fp16 weight-gradient kernel (its one per-layer scale G): word 0 = max|x0|,
        // word k = max|h_k|; they live at the head of the saved buffer, which the compact format leaves unused
        float wm = xmax;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, off));
        if (lane == 0 && wm > 0.f) atomicMax(reinterpret_cast<int*>(p.saved), __float_as_int(wm));
      }
      if (p.saved) {
        // block-transposed copy for the wgrad kernel: [m / 64][field][68]; the two halves write alternate fields
        const size_t m_pad = (size_t)(st * 2 + g) * 128 + t;
        float* xb = p.saved + p.xb_off + (m_pad >> 6) * (size_t)(F * kWgPad) + (m_pad & 63);
        for (int j = q; j < F; j += 2) xb[j * kWgPad] = x0g[((size_t)r * F + j) * D + d];
      }
      for (int k = 0; k < p.n_layers; ++k) {
        const int Hp = p.Hp[k], L = p.L[k];
        const int nh = Hp >> 1;                        // operand values of this thread per granule: 16 or 32
        float srow, inv_row, sw, inv_w;
        tc::pow2_scale_to_1024(xmax * hmax, srow, inv_row);
        tc::pow2_scale_to_1024(__int_as_float(__ldg(p.wmax + k)), sw, inv_w);
        const float inv_acc = inv_row * inv_w;
        for (int i = 0; i < F; ++i) {
          const float xi = x0g[((size_t)r * F + i) * D + d] * srow;
          const uint32_t sa = gran % kT2StagesA, pa = (gran / kT2StagesA) & 1;
          ++gran;
          uint32_t zh[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) zh[c] = tc::pack_f16x2(xi * h[2 * c], xi * h[2 * c + 1]);
          tc::mbar_wait(&empty_a[g * kT2StagesA + sa], pa ^ 1);
          tc::fence_after_thread_sync();
          const uint32_t a_col = tmem_base + lane_base + 2 * kAccCols + (sa * 2 + g) * kT2ACols + q * (nh >> 1);
          tc::tmem_st8v(a_col, zh[0], zh[1], zh[2], zh[3], zh[4], zh[5], zh[6], zh[7]);
          if (nh == 32) tc::tmem_st8v(a_col + 8, zh[8], zh[9], zh[10], zh[11], zh[12], zh[13], zh[14], zh[15]);
          tc::tmem_wait_st();
          tc::fence_before_thread_sync();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&full_a[g * kT2StagesA + sa]);
        }
        // ---- epilogue of layer k: this thread's share of its accumulator row ------------------------------------
        tc::mbar_wait(&acc_full[g], layer_cnt & 1);
        ++layer_cnt;
        tc::fence_after_thread_sync();
        const int hid_n = p.hid_n[k], pool_lo = p.pool_lo[k], pool_n = p.pool_n[k];
        const int nhn = (k + 1 < p.n_layers) ? (p.Hp[k + 1] >> 1) : 0;      // next layer: operand values per thread
        const float* bias = p.bias ? p.bias + p.bias_off[k] : nullptr;
        uint16_t* mrow = (p.saved && p.act == DTB_ACT_RELU && b < p.B)
                             ? reinterpret_cast<uint16_t*>(reinterpret_cast<uint32_t*>(p.saved + p.saved_off[k]) +
                                                           ((size_t)b * D + d) * ((L + 31) >> 5))
                             : nullptr;
        float* hb = nullptr;
        if (p.saved && hid_n > 0) {
          const size_t m_pad = (size_t)(st * 2 + g) * 128 + t;
          hb = p.saved + p.hb_off[k] + (m_pad >> 6) * (size_t)(hid_n * kWgPad) + (m_pad & 63);
        }
        // every granule of this layer has been handed over: h is dead and becomes the next layer's operand in place
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) h[jj] = 0.f;
        // block ownership.  Hidden 16-column blocks (columns < hid_n = the next layer's h): the owner is the half whose
        // operand range [q*nhn, (q+1)*nhn) holds them -- slots 0 and 1 of this thread.  Pooled-only blocks (direct=False:
        // columns [pool_lo, pool_lo + pool_n)): first half of them to q = 0, the rest to q = 1.
        const int first_pb = (pool_lo >= hid_n) ? (pool_lo >> 4) : (hid_n >> 4);     // first block that is pooled but not hidden
        const int last_pb = (pool_lo + pool_n) >> 4;
        const int n_pb = last_pb > first_pb ? last_pb - first_pb : 0;
        const int pb_split = (n_pb + 1) >> 1;
#pragma unroll
        for (int slot = 0; slot < 6; ++slot) {
          // slots 0-1: hidden blocks of this half; slots 2-5: pooled-only blocks of this half
          int cb;
          bool live;
          if (slot < 2) {
            cb = ((q * nhn) >> 4) + slot;
            live = (slot * 16 < nhn) && (cb * 16 < hid_n);
          } else {
            const int s2 = slot - 2;
            cb = first_pb + q * pb_split + s2;
            live = s2 < (q == 0 ? pb_split : n_pb - pb_split);
          }
          if (live) {                                   // warp-uniform
            uint32_t v[16];
            tc::tmem_ld16(tmem_base + lane_base + g * kAccCols + cb * 16, v);
            tc::tmem_wait_ld();
            float o[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float val = __uint_as_float(v[j]) * inv_acc;
              if (bias) val += __ldg(bias + cb * 16 + j);
              if (p.act == DTB_ACT_RELU) val = fmaxf(val, 0.f);
              o[j] = val;
            }
            if (slot < 2) {
#pragma unroll
              for (int j = 0; j < 16; ++j) h[(slot & 1) * 16 + j] = o[j];
              if (hb) {
#pragma unroll
                for (int j = 0; j < 16; ++j) hb[(cb * 16 + j) * kWgPad] = o[j];
              }
            }
            if (mrow) {
              uint32_t bits = 0u;
#pragma unroll
              for (int j = 0; j < 16; ++j) bits |= (o[j] > 0.f ? 1u : 0u) << j;
              mrow[cb] = (uint16_t)bits;
            }
            // sum over the D lanes that share a batch row (reduce-scatter butterfly, see cin_tc_fwd_kernel)
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
        tc::fence_before_thread_sync();
        // ---- next layer's operand: own half of h_{k+1}; row maximum over both halves -----------------------------
        if (k + 1 < p.n_layers) {
          float own = 0.f;
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) own = fmaxf(own, fabsf(h[jj]));
          float* mx = mxg + (size_t)(k & 1) * 2 * 128;
          mx[q * 128 + t] = own;
          asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
          hmax = fmaxf(mx[t], mx[128 + t]);
          if (p.saved && q == 0) {
            float wm = hmax;
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, off));
            if (lane == 0 && wm > 0.f) atomicMax(reinterpret_cast<int*>(p.saved) + k + 1, __float_as_int(wm));
          }
        }
      }
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");   // x0 block free for the next super tile
    }
  } else if (warp < 18) {
    // ================================ MMA issuers: warp 16 -> tile 0, warp 17 -> tile 1 =====================
    // One issuing thread could not keep the tensor pipe fed once the work per granule fell to 8 x 64 cycles: its loop
    // (two barrier waits, ~10 uniform-datapath instructions per UTCHMMA, commits) measured ~720 cycles per granule
    // (ncu source view, profiles/r2_cin_tc2_ncu.txt).  Two warps on different SM sub-partitions each issue one tile.
    const int g = warp - 16;
    const bool leader = elect_one_sync();
    const uint32_t smem_b_u32 = tc::smem_u32(smem_b) + g * kT2StagesB * (uint32_t)p.b_stage_bytes;
    const uint32_t d_tmem = tmem_base + g * kAccCols;
    uint32_t gran = 0, chunk = 0;
    bool go_sent = (g != 0);
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      for (int k = 0; k < p.n_layers; ++k) {
        const int Hp = p.Hp[k], L = p.L[k];
        const uint32_t idesc = tc::make_idesc_f16(128, (uint32_t)L);
        const uint32_t lbo_b = (uint32_t)(L >> 3) * 128;       // K-direction core stride of the W image
        const uint32_t kstep = (2 * lbo_b) >> 4;               // descriptor address units per UMMA k-step
        const uint64_t desc_hi = ((uint64_t)((lbo_b >> 4) & 0x3FFF) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
        for (int i = 0; i < F; ++i, ++chunk, ++gran) {
          const uint32_t sb = chunk % kT2StagesB, pb = (chunk / kT2StagesB) & 1;
          const uint32_t sa = gran % kT2StagesA, pa = (gran / kT2StagesA) & 1;
          const uint32_t a_base = tmem_base + 2 * kAccCols + (sa * 2 + g) * kT2ACols;
          const uint64_t desc0 = desc_hi | (uint64_t)(((smem_b_u32 + sb * (uint32_t)p.b_stage_bytes) >> 4) & 0x3FFF);
          tc::mbar_wait(&full_b[g * kT2StagesB + sb], pb);
          tc::mbar_wait(&full_a[g * kT2StagesA + sa], pa);
          tc::fence_after_thread_sync();
          if (leader) {
            tc::mma_ts(d_tmem, a_base, desc0, idesc, (uint32_t)(i != 0));
            tc::mma_ts(d_tmem, a_base + 8, desc0 + kstep, idesc, 1u);
            if (Hp == 64) {
              tc::mma_ts(d_tmem, a_base + 16, desc0 + 2 * kstep, idesc, 1u);
              tc::mma_ts(d_tmem, a_base + 24, desc0 + 3 * kstep, idesc, 1u);
            }
            tc::mma_commit(&empty_a[g * kT2StagesA + sa]);
            tc::mma_commit(&empty_b[g * kT2StagesB + sb]);
            if (i == F - 1) tc::mma_commit(&acc_full[g]);
            if (!go_sent && (i == F / 2 || i == F - 1)) tc::mma_commit(start1);
          }
          if (i == F / 2 || i == F - 1) go_sent = true;
          __syncwarp();
        }
      }
    }
  } else {
    // ================================ weight loaders: warp 18 -> tile 0's ring, warp 19 -> tile 1's ===============
    const int g = warp - 18;
    if (lane == 0) {
      uint8_t* ring = smem_b + (size_t)g * kT2StagesB * p.b_stage_bytes;
      uint32_t chunk = 0;
      if (g == 1) tc::mbar_wait(start1, 0);
      for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
        for (int k = 0; k < p.n_layers; ++k) {
          const uint32_t bytes = (uint32_t)p.L[k] * p.Hp[k] * 2;       // one fp16 image
          const uint32_t stride = (uint32_t)p.L[k] * p.Hp[k] * 4;      // the pack keeps room for a lo image
          const uint8_t* src = p.wpack + p.wpack_off[k];
          for (int i = 0; i < F; ++i, ++chunk) {
            const uint32_t sb = chunk % kT2StagesB, pb = (chunk / kT2StagesB) & 1;
            tc::mbar_wait(&empty_b[g * kT2StagesB + sb], pb ^ 1);
            tc::mbar_arrive_expect_tx(&full_b[g * kT2StagesB + sb], bytes);
            tc::bulk_g2s(ring + (size_t)sb * p.b_stage_bytes, src + (size_t)i * stride, bytes, &full_b[g * kT2StagesB + sb]);
          }
        }
      }
    }
    __syncwarp();
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 16) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ==========================================================================================
// Backward, data gradient (the counterpart of cin_tc_dgrad_kernel, cin_tc.cu), same two-threads-per-row organisation
// ==========================================================================================
// Per 2 x 128-row super tile, layers last -> first:
//   dC_k = (d_pooled part + dh_{k+1}) * relu'(T_k), scaled per row into fp16 (exact power of two from the row's max, the
//          two halves exchange their maxima) -> TMEM A operand (written ONCE per layer) + fp16 tiles in HBM for wgrad;
//   per x0 field i:  dZ[m, j] = sum_l dC[m, l] W[(i, j), l]      one N = Hp MMA chain, K = L, two accumulators per tile
//   read-out: dx0[m, i] += sum_j dZ h_k[m, j] ;  dh_k[m, j] += dZ x0[m, i]              each thread its half of j
// This kernel is bound by the TMEM read-out of dZ (128 x F*Hp fp32 per tile and layer at ~64 B/clk/SM: ~1.0 ms at
// 65 536 rows), not by the tensor pipe (0.6 ms of MMAs in one fp16 pass; the bf16x3 kernel was MMA-bound at 2.9 ms).
// So the organisation serves the read-out: two 64-column accumulators per tile, the issuing warp one field ahead (the
// MMAs of field i+1 run under the read-out of field i), one issuing warp per tile, the read-out split between two
// threads with 32 + 32 live values each.  (A first version paired two fields per N = 128 chain with ONE accumulator
// per tile: every read-out then waited for its own MMAs -- 1.81 ms, tensor pipe 30 %.)
constexpr int kT2StagesW = 6;          // per-field W images (Hp x L fp16 <= 16 KB each), shared by the two tiles' issuers
// dC tiles handed from the data-gradient to the weight-gradient kernel: blocks of 16 GEMM rows,
// [fp16 image, MN-major: (l / 8) groups of 256 B = 2 k-groups x 8 rows x 16 B | 16 floats 1 / t_m]
__host__ __device__ inline size_t tc2_dc_blk(int L) { return (size_t)32 * L + 64; }

struct T2BwdSmem {
  int b_off, x0_off, dx_off, mx_off, bar_off, total;
};
__host__ __device__ inline T2BwdSmem tc2_bwd_layout(int b_stage_bytes, int F) {
  T2BwdSmem l;
  l.b_off = 0;
  l.x0_off = kT2StagesW * b_stage_bytes;
  l.dx_off = l.x0_off + 2 * 128 * F * 4;           // x0s[tile][r][i][d]
  l.mx_off = l.dx_off + 2 * 2 * 128 * F * 4;       // dxs[tile][half][i][t]
  l.bar_off = l.mx_off + 2 * 2 * 2 * 128 * 4;      // row maxima [tile][parity][half][t]
  l.bar_off = (l.bar_off + 15) / 16 * 16;
  l.total = l.bar_off + 256;
  return l;
}

// max |d_pooled[b, pooled columns of layer k]| per batch row and layer: the data-gradient kernel scales each dC row
// into fp16 by a power of two taken from an UPPER BOUND of the row's maximum (this + max|dh|), so that it needs one
// sweep over the row instead of two.  One warp per batch row.
struct DpmaxTab {
  int pcol0[kCinMaxLayers], pool_n[kCinMaxLayers];
};
__global__ void cin_tc2_dpmax_kernel(const float* __restrict__ d_pooled, float* __restrict__ out, int B, int P, int n_layers,
                                     const DpmaxTab tab) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int b = warp; b < B; b += n_warps) {
    const float* row = d_pooled + (size_t)b * P;
    for (int k = 0; k < n_layers; ++k) {
      float m = 0.f;
      for (int c = lane; c < tab.pool_n[k]; c += 32) m = fmaxf(m, fabsf(__ldg(row + tab.pcol0[k] + c)));
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
      if (lane == 0) out[(size_t)b * n_layers + k] = m;
    }
  }
}

template <int D>
__global__ void __launch_bounds__(kT2Threads, 1) cin_tc2_dgrad_kernel(const __grid_constant__ CinTcBwdParams p) {
  constexpr int R = 128 / D;
  extern __shared__ __align__(1024) uint8_t smem[];
  const T2BwdSmem lay = tc2_bwd_layout(p.b_stage_bytes, p.F);
  uint8_t* smem_b = smem + lay.b_off;
  float* x0s = reinterpret_cast<float*>(smem + lay.x0_off);
  float* dxs = reinterpret_cast<float*>(smem + lay.dx_off);
  float* mxs = reinterpret_cast<float*>(smem + lay.mx_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* a_ready = bars;          // [tile]        8 warps
  uint64_t* full_b = bars + 2;       // [stage]       bulk copy (tx)
  uint64_t* empty_b = bars + 8;      // [stage]       one commit per issuing warp
  uint64_t* acc_full = bars + 14;    // [tile][buf]   commit
  uint64_t* acc_empty = bars + 18;   // [tile][buf]   8 warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = p.F;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);

  if (threadIdx.x == 0) {
    for (int g = 0; g < 2; ++g) tc::mbar_init(&a_ready[g], 8);
    for (int i = 0; i < 4; ++i) {
      tc::mbar_init(&acc_full[i], 1);
      tc::mbar_init(&acc_empty[i], 8);
    }
    for (int s = 0; s < kT2StagesW; ++s) {
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty_b[s], 2);
    }
    tc::fence_barrier_init();
  }
  if (warp == 16) tc::tmem_alloc(tmem_slot, kTmemCols);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 16) {
    const int g = warp >> 3, q = (warp >> 2) & 1;
    const int t = (warp & 3) * 32 + lane;
    const int tt = q * 128 + t;
    const int r = t / D, d = t % D;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t t_tile = tmem_base + lane_base + g * 256;   // A: columns [0, 64) ; accumulator: [64, 192)
    float* x0g = x0s + (size_t)g * 128 * F;                     // [r][i][d]
    float* dxg = dxs + ((size_t)g * 2 + q) * 128 * F;           // [i][t]  this half's partial dx0
    float* dxo = dxs + ((size_t)g * 2 + (q ^ 1)) * 128 * F;     //         the other half's
    float* mxg = mxs + (size_t)g * 2 * 2 * 128;                 // [parity][half][t]
    uint32_t acc_cnt = 0, mx_cnt = 0;
    float h[32], dh[32];
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      const int row0 = (st * 2 + g) * R;
      const int b = row0 + r;
      const bool valid = b < p.B;
      const size_t m_pad = (size_t)(st * 2 + g) * 128 + t;      // == b*D + d
      {
        constexpr int Q = D / 4;
        for (int e = tt; e < R * F * Q; e += 256) {
          const int rr = e / (F * Q);
          const int rem = e - rr * F * Q;
          const int i = rem / Q, qq = rem - i * Q;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row0 + rr < p.B) {
            const int64_t rb = table_row(p.row_offsets, i, __ldg(p.idx + (int64_t)(row0 + rr) * F + i), D, nullptr);
            if (rb >= 0) v = ldg_stream_f4(p.table + rb + (qq << 2));
          }
          *reinterpret_cast<float4*>(x0g + ((size_t)rr * F + i) * D + (qq << 2)) = v;
        }
        for (int i = 0; i < F; ++i) dxg[i * 128 + t] = 0.f;
      }
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) dh[jj] = 0.f;
      float dhmax = 0.f;                                         // max |dh row| over both halves (gradient wrt h_{k+1})
      for (int k = p.n_layers - 1; k >= 0; --k) {
        const int L = p.L[k], Hp = p.Hp[k];
        const int nh = Hp >> 1;                                              // this thread's share of j: 16 or 32
        const int hid_n = p.hid_n[k], pool_lo = p.pool_lo[k], pool_n = p.pool_n[k];
        const int nhn = (k + 1 < p.n_layers) ? (p.Hp[k + 1] >> 1) : 0;      // the next layer's share (dh holds its gradient)
        const int first_pb = (pool_lo >= hid_n) ? (pool_lo >> 4) : (hid_n >> 4);
        const int last_pb = (pool_lo + pool_n) >> 4;
        const int n_pb = last_pb > first_pb ? last_pb - first_pb : 0;
        const int pb_split = (n_pb + 1) >> 1;
        const uint16_t* mrow = (p.act == DTB_ACT_RELU && valid)
                                   ? reinterpret_cast<const uint16_t*>(reinterpret_cast<const uint32_t*>(p.saved + p.saved_off[k]) +
                                                                       m_pad * ((L + 31) >> 5))
                                   : nullptr;
        const float* dprow = p.d_pooled + (size_t)b * p.P + p.pcol0[k];
        // ---- row scale from an upper bound of max|dC_k row|: max|d_pooled part| (precomputed per batch row) + max|dh| ------
        float trow, inv_t;
        const float bound = (valid ? __ldg(p.dpmax + (size_t)b * p.n_layers + k) : 0.f) + dhmax;
        tc::pow2_scale_to_1024(bound, trow, inv_t);
        if (q == 0) {
          // wgrad folds 1/t_m into its on-the-fly operand: one float per row in the unused "lo" slot of the row's
          // 16-row tile block; the layer's max|dC| bound goes to the statistics words (slot 8 + k)
          // a row whose bound is zero has dC == 0: it must contribute NOTHING.  With 1/t_m = 1 (the scale of a zero bound)
          // its operand x0 h G would overflow fp16 to inf and inf * 0 = NaN poisoned the whole filter gradient (found
          // on the five-net config, where rows with an exactly zero upstream gradient exist)
          *reinterpret_cast<float*>(p.dc_tiles + p.dc_off[k] + (m_pad >> 4) * tc2_dc_blk(L) + 32 * L + (t & 15) * 4) =
              bound > 0.f ? inv_t : 0.f;
          float wm = bound;
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, off));
          if (lane == 0 && wm > 0.f) atomicMax(const_cast<int*>(p.wmax) + 8 + k, __float_as_int(wm));
        }
        // ---- the 16-column blocks of dC_k this thread owns (same rule as the forward's read-out): one sweep ---------------
        uint8_t* dcblk = p.dc_tiles + p.dc_off[k] + (m_pad >> 4) * tc2_dc_blk(L) + ((t & 15) >> 3) * 128 + (t & 7) * 16;
#pragma unroll
        for (int slot = 0; slot < 6; ++slot) {
          int cb;
          bool live;
          if (slot < 2) {
            cb = ((q * nhn) >> 4) + slot;
            live = (slot * 16 < nhn) && (cb * 16 < hid_n);
          } else {
            const int s2 = slot - 2;
            cb = first_pb + q * pb_split + s2;
            live = s2 < (q == 0 ? pb_split : n_pb - pb_split);
          }
          if (live) {                               // warp-uniform
            float dc[16];
            const int pc = cb * 16 - pool_lo;       // first pooled column of the block (blocks never straddle the range)
            if (valid && pc >= 0 && pc < pool_n) {
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                const float4 q4 = __ldg(reinterpret_cast<const float4*>(dprow + pc + j));
                dc[j] = q4.x; dc[j + 1] = q4.y; dc[j + 2] = q4.z; dc[j + 3] = q4.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) dc[j] = 0.f;
            }
            if (slot < 2) {
#pragma unroll
              for (int j = 0; j < 16; ++j) dc[j] += dh[(slot & 1) * 16 + j];
            }
            uint32_t keep = valid ? 0xffffu : 0u;
            if (mrow) keep = (uint32_t)__ldg(mrow + cb);
            else if (p.act == DTB_ACT_RELU) keep = 0u;                  // padded row
            uint32_t zf[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float lo = ((keep >> (2 * c)) & 1u) ? dc[2 * c] * trow : 0.f;
              const float hi = ((keep >> (2 * c + 1)) & 1u) ? dc[2 * c + 1] * trow : 0.f;
              zf[c] = tc::pack_f16x2(lo, hi);
            }
            tc::tmem_st8v(t_tile + cb * 8, zf[0], zf[1], zf[2], zf[3], zf[4], zf[5], zf[6], zf[7]);
            *reinterpret_cast<uint4*>(dcblk + (cb * 2) * 256) = make_uint4(zf[0], zf[1], zf[2], zf[3]);
            *reinterpret_cast<uint4*>(dcblk + (cb * 2 + 1) * 256) = make_uint4(zf[4], zf[5], zf[6], zf[7]);
            tc::tmem_wait_st();                                         // zf is reused by the next block
          }
        }
        tc::fence_before_thread_sync();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&a_ready[g]);
        float sw, inv_w;
        tc::pow2_scale_to_1024(__int_as_float(__ldg(p.wmax + k)), sw, inv_w);
        const float inv_acc = inv_t * inv_w;
        // ---- this thread's half of h_k, and a fresh dh accumulator ------------------------------------------------
        if (k > 0) {
          const int Hk = p.H[k];
          const float* hbp = p.saved + p.hb_off[k - 1] + (m_pad >> 6) * (size_t)(Hk * kWgPad) + (m_pad & 63);
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const int j = q * nh + jj;
            h[jj] = (valid && jj < nh && j < Hk) ? __ldg(hbp + (size_t)j * kWgPad) : 0.f;
          }
        } else {
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const int j = q * nh + jj;
            h[jj] = (jj < nh && j < F) ? x0g[((size_t)r * F + j) * D + d] : 0.f;
          }
        }
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) dh[jj] = 0.f;
        for (int i = 0; i < F; ++i) {
          const uint32_t buf = acc_cnt & 1, par = (acc_cnt >> 1) & 1;
          ++acc_cnt;
          const float xi = x0g[((size_t)r * F + i) * D + d] * inv_acc;
          tc::mbar_wait(&acc_full[g * 2 + buf], par);
          tc::fence_after_thread_sync();
          float dx = 0.f;
#pragma unroll
          for (int blk = 0; blk < 2; ++blk) {
            if (blk * 16 < nh) {
              uint32_t v[16];
              tc::tmem_ld16(t_tile + 64 + buf * 64 + q * nh + blk * 16, v);
              tc::tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float dz = __uint_as_float(v[j]);
                dx = fmaf(dz, h[blk * 16 + j], dx);
                dh[blk * 16 + j] = fmaf(dz, xi, dh[blk * 16 + j]);
              }
            }
          }
          tc::fence_before_thread_sync();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&acc_empty[g * 2 + buf]);
          dxg[i * 128 + t] += dx * inv_acc;
        }
        if (k == 0) {
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const int j = q * nh + jj;
            if (jj < nh && j < F) dxg[j * 128 + t] += dh[jj];     // h_0 is x0 itself
          }
        } else {
          // max |dh_k row| over both halves: the bound of the next (lower) layer's dC
          float own = 0.f;
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) own = fmaxf(own, fabsf(dh[jj]));
          float* mx = mxg + (size_t)(mx_cnt & 1) * 2 * 128;
          ++mx_cnt;
          mx[q * 128 + t] = own;
          asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
          dhmax = fmaxf(mx[t], mx[128 + t]);
        }
      }
      // ---- scatter dx0 of this tile into the embedding gradient: both halves' partial sums, alternate fields ----------
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
      if (valid) {
        for (int i = q; i < F; i += 2) {
          const int64_t rb = table_row(p.row_offsets, i, __ldg(p.idx + (int64_t)b * F + i), D, nullptr);
          if (rb >= 0) atomicAdd(p.grad_table + rb + d, dxg[i * 128 + t] + dxo[i * 128 + t]);
        }
      }
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
    }
  } else if (warp < 18) {
    // ---- MMA issuers: warp 16 -> tile 0, warp 17 -> tile 1 (independent ping-pong partners) ----------------------------
    const int g = warp - 16;
    const bool leader = elect_one_sync();
    const uint32_t smem_b_u32 = tc::smem_u32(smem_b);
    const uint32_t a_base = tmem_base + g * 256;
    uint32_t chunk = 0, cnt = 0, layer_cnt = 0;
    for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
      for (int k = p.n_layers - 1; k >= 0; --k, ++layer_cnt) {
        const int Hp = p.Hp[k], L = p.L[k];
        const uint32_t idesc = tc::make_idesc_f16(128, (uint32_t)Hp);
        const uint32_t lbo_b = (uint32_t)(Hp >> 3) * 128;
        const uint32_t kstep = (2 * lbo_b) >> 4;
        const uint64_t desc_hi = ((uint64_t)((lbo_b >> 4) & 0x3FFF) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
        for (int i = 0; i < F; ++i, ++chunk, ++cnt) {
          const uint32_t sb = chunk % kT2StagesW, pb = (chunk / kT2StagesW) & 1;
          const uint32_t buf = cnt & 1, par = (cnt >> 1) & 1;
          const uint64_t desc0 = desc_hi | (uint64_t)(((smem_b_u32 + sb * (uint32_t)p.b_stage_bytes) >> 4) & 0x3FFF);
          const uint32_t d_tmem = a_base + 64 + buf * 64;
          tc::mbar_wait(&full_b[sb], pb);
          if (i == 0) tc::mbar_wait(&a_ready[g], layer_cnt & 1);
          tc::mbar_wait(&acc_empty[g * 2 + buf], par ^ 1);
          tc::fence_after_thread_sync();
          if (leader) {
#pragma unroll
            for (int ks = 0; ks < kMaxL / 16; ++ks)
              if (ks * 16 < L) tc::mma_ts(d_tmem, a_base + ks * 8, desc0 + ks * kstep, idesc, (uint32_t)(ks != 0));
            tc::mma_commit(&acc_full[g * 2 + buf]);
            tc::mma_commit(&empty_b[sb]);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 18) {
    if (lane == 0) {
      uint32_t chunk = 0;
      for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
        for (int k = p.n_layers - 1; k >= 0; --k) {
          const uint32_t bytes = (uint32_t)p.Hp[k] * (uint32_t)p.L[k] * 2u;         // one fp16 image (cin_tc_pack_t_f16_kernel)
          const uint32_t stride = (uint32_t)p.Hp[k] * (uint32_t)p.L[k] * 4u;        // the pack keeps room for a lo image
          const uint8_t* src = p.wpack + p.wpack_off[k];
          for (int i = 0; i < F; ++i, ++chunk) {
            const uint32_t sb = chunk % kT2StagesW, pb = (chunk / kT2StagesW) & 1;
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
  if (warp == 16) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// d_bias[l] += sum over rows of dC, from the fp16 tiles (row m scaled by t_m, 1/t_m stored behind the image)
__global__ void cin_tc2_dbias_kernel(const uint8_t* __restrict__ dc_tiles, float* __restrict__ d_bias, int L, int n_blocks16) {
  const int64_t total = (int64_t)n_blocks16 * L;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t blk = t / L;
    const int l = (int)(t - blk * L);
    const uint8_t* base = dc_tiles + blk * (int64_t)tc2_dc_blk(L);
    const uint8_t* col = base + (l >> 3) * 256 + (l & 7) * 2;
    const float* inv_t = reinterpret_cast<const float*>(base + 32 * L);
    float s = 0.f;
    for (int m = 0; m < 16; ++m)
      s += __half2float(*reinterpret_cast<const __half*>(col + (m >> 3) * 128 + (m & 7) * 16)) * __ldg(inv_t + m);
    if (s != 0.f) atomicAdd(d_bias + l, s);
  }
}

// ==========================================================================================
// Backward, weight gradient on ONE fp16 pass
// ==========================================================================================
//   dW_k[(i,j), l] = sum_m x0[m,i] h_k[m,j] dC_k[m,l]     UMMA M = (i,j) pairs, K = batch x dim rows m, N = L
// The reduction runs over m, so per-row scales must cancel inside the MMA: the dC tile row m carries t_m, the
// on-the-fly operand A'[(i,j), m] = x0[m,i] h[m,j] (G / t_m) its inverse and ONE per-layer G (from the recorded maxima)
// keeps |A'| < 1024.  What changed against a first fp16 version built like cin_tc_wgrad_kernel (removed, in git history
// at commit 021caee; 1.94 ms for the three layers, tensor pipe 32 %, producers issue-bound: 3 multiplies + operand
// fetches per element in 256 threads):
//   * a SCALER warp multiplies the x0 tile of a stage by G / t_m once (F x 64 products) -- the 256 producer threads then
//     do ONE multiply per element (x' h) instead of three;
//   * one MMA-issuing warp per tile; 4 operand stages (an fp16 operand block is 32 TMEM columns, not 64);
//   * dC blocks without the unused "lo" half: 16.6 KB per 64-row stage instead of 32 KB from L2.
constexpr int kW2Threads = 448;       // warps 0-7 producers (+ epilogue), 8/9 MMA issue tile 0/1, 10 dC loader, 11 x0/h loader, 12/13 scalers
constexpr int kW2Stages = 3;          // x0 / h / dC stages of 64 rows
constexpr int kW2StagesA = 4;         // operand blocks in TMEM per tile

struct CinTc2WgradParams {
  const float* xb;           // block-transposed x0:  [M_pad/64][F][68]
  const float* hb;           // block-transposed h_k: [M_pad/64][H][68]  (== xb for layer 0)
  const uint8_t* dc_tiles;   // layer k blocks of 16 rows (tc2_dc_blk)
  float* d_w;                // [F*H, L] accumulate
  int F, H, Hp, L;
  int n_stage_total;         // ceil(M_pad / 64)
  int stages_per_split;
  const int* stats;          // [8 + k] max|dC_k| bound, [16] max|x0|, [24 + k] max|h_k| (bit patterns)
  int layer;
};

struct W2Smem {
  int b_off, h_off, x_off, xs_off, bar_off, total, b_bytes, h_bytes, x_bytes;
};
__host__ __device__ inline W2Smem w2_layout(int L, int Hp, int F) {
  W2Smem l;
  l.b_bytes = 4 * (int)tc2_dc_blk(L);
  l.h_bytes = Hp * kWgPad * 4;
  l.x_bytes = F * kWgPad * 4;
  l.b_off = 0;
  l.h_off = kW2Stages * l.b_bytes;
  l.x_off = l.h_off + kW2Stages * l.h_bytes;
  l.xs_off = l.x_off + kW2Stages * l.x_bytes;
  l.bar_off = l.xs_off + kW2Stages * l.x_bytes;
  l.bar_off = (l.bar_off + 15) / 16 * 16;
  l.total = l.bar_off + 320;                      // 32 mbarriers + the TMEM address slot
  return l;
}

__global__ void __launch_bounds__(kW2Threads, 1) cin_tc2_wgrad_kernel(const __grid_constant__ CinTc2WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const W2Smem lay = w2_layout(p.L, p.Hp, p.F);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* full_b = bars;            // [stage] 3   dC blocks landed (tx)
  uint64_t* empty_b = bars + 3;       // [stage] 3   both issuers done with them (+ the scaler read 1/t_m)
  uint64_t* full_h = bars + 6;        // [stage] 3   x0 / h tiles landed (tx)
  uint64_t* scaled = bars + 9;        // [stage] 3   scaler wrote x0 * G / t_m
  uint64_t* empty_h = bars + 12;      // [stage] 3   8 producer warps done reading the tiles
  uint64_t* full_a = bars + 15;       // [tile][stageA] 8
  uint64_t* empty_a = bars + 23;      // [tile][stageA] 8
  uint64_t* acc_done = bars + 31;     // 1 (count 2)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + lay.bar_off + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = p.F, H = p.H, Hp = p.Hp, L = p.L;
  const int ipt = 128 / Hp;                              // x0 fields per 128-row tile
  const int s_begin = blockIdx.y * p.stages_per_split;
  int s_end = s_begin + p.stages_per_split;
  if (s_end > p.n_stage_total) s_end = p.n_stage_total;
  const int n_st = s_end > s_begin ? s_end - s_begin : 0;
  const bool h_is_x = (p.hb == p.xb);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kW2Stages; ++s) {
      tc::mbar_init(&full_b[s], 1);
      tc::mbar_init(&empty_b[s], 4);          // two issuers + two scalers
      tc::mbar_init(&full_h[s], 1);
      tc::mbar_init(&scaled[s], 2);
      tc::mbar_init(&empty_h[s], 8);
    }
    for (int i = 0; i < 2 * kW2StagesA; ++i) {
      tc::mbar_init(&full_a[i], 4);
      tc::mbar_init(&empty_a[i], 1);
    }
    tc::mbar_init(acc_done, 2);
    tc::fence_barrier_init();
  }
  if (warp == 8) tc::tmem_alloc(tmem_slot, kTmemCols);
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;

  float gscale, inv_g;
  {
    const float xm = __int_as_float(__ldg(p.stats + 16)), hm = __int_as_float(__ldg(p.stats + 24 + p.layer));
    const float dm = __int_as_float(__ldg(p.stats + 8 + p.layer));
    tc::pow2_scale_to_1024(xm * hm * dm * (1.0f / 512.0f), gscale, inv_g);     // 1/t_m <= max|dC| / 512
  }

  if (warp < 8) {
    // ---- A producers: lane row = (il, j): A'[row, m] = x'[m, i] * h[m, j] ------------------------------------------
    const int g = warp >> 2;
    const int t = threadIdx.x & 127;
    // GEMM row t <-> (hidden field j = t / ipt, x0 field il = t % ipt): the ipt lanes that share j read the same h row
    // (one 16-byte segment per group instead of one per lane).  This kernel is shared-memory bound -- every product
    // needs two operands from the stage tiles -- and with the (il, j) order of cin_tc_wgrad_kernel a warp's h reads took
    // 4 wavefronts per LDS.128; now 32 / ipt distinct segments = 2 (Hp = 64) or 1 (Hp = 32).
    const int il = t % ipt, j = t / ipt;
    const int i = (blockIdx.x * 2 + g) * ipt + il;
    const bool live = (i < F) && (j < H);
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    for (int s = 0; s < n_st; ++s) {
      const uint32_t sh = s % kW2Stages, ph = (s / kW2Stages) & 1;
      const uint32_t sa = s % kW2StagesA, pa = (s / kW2StagesA) & 1;
      const float* xs = reinterpret_cast<const float*>(smem + lay.xs_off + sh * lay.x_bytes);       // scaled x0 tile
      const float* hs = h_is_x ? reinterpret_cast<const float*>(smem + lay.x_off + sh * lay.x_bytes)
                               : reinterpret_cast<const float*>(smem + lay.h_off + sh * lay.h_bytes);
      tc::mbar_wait(&scaled[sh], ph);               // implies full_h and full_b
      const float4* xrow = reinterpret_cast<const float4*>(xs + (live ? i : 0) * kWgPad);
      const float4* hrow = reinterpret_cast<const float4*>(hs + (live ? j : 0) * kWgPad);
      uint32_t zh[32];
#pragma unroll
      for (int q4 = 0; q4 < 16; ++q4) {
        const float4 xv = xrow[q4], hv = hrow[q4];
        zh[2 * q4] = live ? tc::pack_f16x2(xv.x * hv.x, xv.y * hv.y) : 0u;
        zh[2 * q4 + 1] = live ? tc::pack_f16x2(xv.z * hv.z, xv.w * hv.w) : 0u;
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&empty_h[sh]);
      tc::mbar_wait(&empty_a[g * kW2StagesA + sa], pa ^ 1);
      tc::fence_after_thread_sync();
      const uint32_t a_col = tmem_base + lane_base + 256 + (g * kW2StagesA + sa) * 32;     // 8 columns per k-step
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)
        tc::tmem_st8v(a_col + ks * 8, zh[ks * 8 + 0], zh[ks * 8 + 1], zh[ks * 8 + 2], zh[ks * 8 + 3], zh[ks * 8 + 4],
                      zh[ks * 8 + 5], zh[ks * 8 + 6], zh[ks * 8 + 7]);
      tc::tmem_wait_st();
      tc::fence_before_thread_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&full_a[g * kW2StagesA + sa]);
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
            for (int c = 0; c < 16; ++c) atomicAdd(dst + cb * 16 + c, __uint_as_float(v[c]) * inv_g);
          }
        }
      }
      tc::fence_before_thread_sync();
    }
  } else if (warp < 10) {
    // ---- MMA issuers: warp 8 -> tile 0, warp 9 -> tile 1 -------------------------------------------------------------
    const int g = warp - 8;
    const bool leader = elect_one_sync();
    const uint32_t idesc = tc::make_idesc_f16(128, (uint32_t)L) | (1u << 16);       // B operand MN-major
    // dC block descriptor (MN-major): LBO = 128 B (k-group), SBO = 256 B (n-group)
    const uint64_t desc_hi = ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
    const uint32_t smem_b_u32 = tc::smem_u32(smem + lay.b_off);
    const uint32_t blk16 = (uint32_t)tc2_dc_blk(L) >> 4;
    const uint32_t d_tmem = tmem_base + g * kAccCols;
    for (int s = 0; s < n_st; ++s) {
      const uint32_t sb = s % kW2Stages, pb = (s / kW2Stages) & 1;
      const uint32_t sa = s % kW2StagesA, pa = (s / kW2StagesA) & 1;
      const uint64_t desc0 = desc_hi | (uint64_t)(((smem_b_u32 + sb * (uint32_t)lay.b_bytes) >> 4) & 0x3FFF);
      const uint32_t a_base = tmem_base + 256 + (g * kW2StagesA + sa) * 32;
      tc::mbar_wait(&full_b[sb], pb);
      tc::mbar_wait(&full_a[g * kW2StagesA + sa], pa);
      tc::fence_after_thread_sync();
      if (leader) {
        tc::mma_ts(d_tmem, a_base, desc0, idesc, (uint32_t)(s != 0));
        tc::mma_ts(d_tmem, a_base + 8, desc0 + blk16, idesc, 1u);
        tc::mma_ts(d_tmem, a_base + 16, desc0 + 2 * blk16, idesc, 1u);
        tc::mma_ts(d_tmem, a_base + 24, desc0 + 3 * blk16, idesc, 1u);
        tc::mma_commit(&empty_a[g * kW2StagesA + sa]);
        tc::mma_commit(&empty_b[sb]);
        if (s == n_st - 1) tc::mma_commit(acc_done);
      }
      __syncwarp();
    }
  } else if (warp == 10) {
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)lay.b_bytes;
      for (int s = 0; s < n_st; ++s) {
        const uint32_t sb = s % kW2Stages, pb = (s / kW2Stages) & 1;
        tc::mbar_wait(&empty_b[sb], pb ^ 1);
        tc::mbar_arrive_expect_tx(&full_b[sb], bytes);
        tc::bulk_g2s(smem + lay.b_off + sb * lay.b_bytes, p.dc_tiles + (size_t)(s_begin + s) * bytes, bytes, &full_b[sb]);
      }
    }
    __syncwarp();
  } else if (warp == 11) {
    // ---- x0 / h tile loader: one bulk async copy each per 64-row stage ---------------------------------------------
    if (lane == 0) {
      const uint32_t x_bytes = (uint32_t)lay.x_bytes, h_bytes = (uint32_t)(H * kWgPad * 4);
      for (int s = 0; s < n_st; ++s) {
        const uint32_t sh = s % kW2Stages, ph = (s / kW2Stages) & 1;
        tc::mbar_wait(&empty_h[sh], ph ^ 1);
        const size_t blk = (size_t)(s_begin + s);
        tc::mbar_arrive_expect_tx(&full_h[sh], x_bytes + (h_is_x ? 0u : h_bytes));
        tc::bulk_g2s(smem + lay.x_off + sh * lay.x_bytes, p.xb + blk * (size_t)(F * kWgPad), x_bytes, &full_h[sh]);
        if (!h_is_x)
          tc::bulk_g2s(smem + lay.h_off + sh * lay.h_bytes, p.hb + blk * (size_t)(H * kWgPad), h_bytes, &full_h[sh]);
      }
    }
    __syncwarp();
  } else {
    // ---- scalers (warps 12, 13: even / odd fields): x'[i][m] = x0[i][m] * G / t_m for the 64 rows of the stage; a lane
    //      owns rows 2 lane and 2 lane + 1 (8-byte accesses) ------------------------------------------------------------
    const int sw = warp - 12;
    for (int s = 0; s < n_st; ++s) {
      const uint32_t sh = s % kW2Stages, ph = (s / kW2Stages) & 1;
      tc::mbar_wait(&full_h[sh], ph);
      tc::mbar_wait(&full_b[sh], ph);
      const uint8_t* bst = smem + lay.b_off + sh * lay.b_bytes;
      const float2 c = *reinterpret_cast<const float2*>(bst + (lane >> 3) * tc2_dc_blk(L) + 32 * L + (lane & 7) * 8);
      const float c0 = c.x * gscale, c1 = c.y * gscale;
      const float* xs = reinterpret_cast<const float*>(smem + lay.x_off + sh * lay.x_bytes);
      float* xd = reinterpret_cast<float*>(smem + lay.xs_off + sh * lay.x_bytes);
      // 8 fields at a time with all loads in flight (a rolled loop made this warp the kernel's bottleneck)
      for (int i0 = sw; i0 < F; i0 += 16) {
        float2 a[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + 2 * u < F ? i0 + 2 * u : sw;
          a[u] = *reinterpret_cast<const float2*>(xs + i * kWgPad + 2 * lane);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (i0 + 2 * u < F)
            *reinterpret_cast<float2*>(xd + (i0 + 2 * u) * kWgPad + 2 * lane) = make_float2(a[u].x * c0, a[u].y * c1);
      }
      __syncwarp();
      if (lane == 0) {
        tc::mbar_arrive(&scaled[sh]);
        tc::mbar_arrive(&empty_b[sh]);         // the 1/t_m words have been read
      }
    }
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  if (warp == 8) {
    tc::fence_after_thread_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int tc2_b_stage(const CinTcParams& p) {
  int b = 0;
  for (int k = 0; k < p.n_layers; ++k) {
    const int bytes = p.L[k] * p.Hp[k] * 2;
    if (bytes > b) b = bytes;
  }
  return b;
}

bool cin_tc2_fwd_supported(const CinTcParams& p, int D) {
  if (D != 16 && D != 32) return false;
  if (p.n_pass != 1) return false;
  if (p.saved && !p.compact) return false;             // the full (fp32 T_k) saved format is written by cin_tc_fwd_kernel only
  for (int k = 0; k < p.n_layers; ++k) {
    if (p.Hp[k] != 32 && p.Hp[k] != 64) return false;
    if (p.L[k] % 16 || p.L[k] > kMaxL) return false;
    if (p.hid_n[k] % 16 || p.pool_lo[k] % 16 || p.pool_n[k] % 16) return false;
    if (p.hid_n[k] > 0 && p.pool_lo[k] != 0 && p.pool_lo[k] != p.hid_n[k]) return false;
  }
  return tc2_layout(tc2_b_stage(p), p.F).total <= 227 * 1024;
}

template <int D>
static int tc2_launch(const CinTcParams& p_in, cudaStream_t st) {
  CinTcParams p = p_in;
  p.b_stage_bytes = tc2_b_stage(p);
  const T2Smem lay = tc2_layout(p.b_stage_bytes, p.F);
  auto kern = cin_tc2_fwd_kernel<D>;
  DTB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, lay.total));
  if (p.saved) DTB_CUDA_OK(cudaMemsetAsync(p.saved, 0, 64, st));          // operand maxima words (see the kernel)
  const int R = 128 / D;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);
  int grid = sm_count();
  if (grid > n_super) grid = n_super;
  kern<<<grid, kT2Threads, lay.total, st>>>(p);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

static int tc2_bwd_b_stage(const CinTcBwdParams& p) {
  int b = 0;
  for (int k = 0; k < p.n_layers; ++k) {
    const int bytes = p.Hp[k] * p.L[k] * 2;
    if (bytes > b) b = bytes;
  }
  return b;
}

bool cin_tc2_bwd_supported(const CinTcBwdParams& p, int D) {
  if (D != 16 && D != 32) return false;
  if (!p.compact) return false;
  for (int k = 0; k < p.n_layers; ++k) {
    if (p.Hp[k] != 32 && p.Hp[k] != 64) return false;
    if (p.L[k] % 16 || p.L[k] > kMaxL) return false;
    if (p.hid_n[k] % 16 || p.pool_lo[k] % 16 || p.pool_n[k] % 16) return false;
    if (p.hid_n[k] > 0 && p.pool_lo[k] != 0 && p.pool_lo[k] != p.hid_n[k]) return false;
    if (!cin_tc2_wgrad_supported(p.F, p.Hp[k], p.L[k])) return false;
  }
  return tc2_bwd_layout(tc2_bwd_b_stage(p), p.F).total <= 227 * 1024;
}

template <int D>
static int tc2_launch_dgrad(const CinTcBwdParams& p_in, cudaStream_t st) {
  CinTcBwdParams p = p_in;
  p.b_stage_bytes = tc2_bwd_b_stage(p);
  const T2BwdSmem lay = tc2_bwd_layout(p.b_stage_bytes, p.F);
  auto kern = cin_tc2_dgrad_kernel<D>;
  DTB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, lay.total));
  const int R = 128 / D;
  const int n_super = (p.B + 2 * R - 1) / (2 * R);
  int grid = sm_count();
  if (grid > n_super) grid = n_super;
  kern<<<grid, kT2Threads, lay.total, st>>>(p);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

// per-(batch row, layer) max|d_pooled| -> out[B, n_layers]
int cin_tc2_dpmax(const float* d_pooled, float* out, const int* pcol0_host, const int* pool_n_host, int B, int P, int n_layers,
                  cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(d_pooled) & 15) || (P & 3)) {
    set_error("dtb_cin_bwd: fp16 single pass needs d_pooled 16-byte aligned with a row length divisible by 4");
    return DTB_ERR_INVALID_ARG;
  }
  DpmaxTab tab{};
  for (int k = 0; k < n_layers; ++k) {
    tab.pcol0[k] = pcol0_host[k];
    tab.pool_n[k] = pool_n_host[k];
  }
  int blocks = (B + 7) / 8;
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  cin_tc2_dpmax_kernel<<<blocks, 256, 0, st>>>(d_pooled, out, B, P, n_layers, tab);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int cin_tc2_launch_dgrad(const CinTcBwdParams& p, int D, cudaStream_t st) {
  if (D == 16) return tc2_launch_dgrad<16>(p, st);
  if (D == 32) return tc2_launch_dgrad<32>(p, st);
  set_error("cin_tc2: embedding dim %d unsupported", D);
  return DTB_ERR_UNSUPPORTED;
}

int cin_tc2_dbias(const uint8_t* dc_tiles, float* d_bias, int L, int n_blocks16, cudaStream_t st) {
  int blocks = (int)(((int64_t)n_blocks16 * L + 255) / 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  cin_tc2_dbias_kernel<<<blocks, 256, 0, st>>>(dc_tiles, d_bias, L, n_blocks16);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

bool cin_tc2_wgrad_supported(int F, int Hp, int L) { return w2_layout(L, Hp, F).total <= 227 * 1024 && (Hp == 32 || Hp == 64); }

// one layer: xb / hb block-transposed operand tiles, dc_tiles the layer's fp16 blocks, d_w accumulated
int cin_tc2_launch_wgrad(const float* xb, const float* hb, const uint8_t* dc_tiles, float* d_w, int F, int H, int Hp, int L,
                         int n_stage_total, const int* stats, int layer, cudaStream_t st) {
  CinTc2WgradParams w{};
  w.xb = xb; w.hb = hb; w.dc_tiles = dc_tiles; w.d_w = d_w;
  w.F = F; w.H = H; w.Hp = Hp; w.L = L; w.n_stage_total = n_stage_total; w.stats = stats; w.layer = layer;
  const int ipt = 128 / Hp;
  const int n_tiles = (F + ipt - 1) / ipt;
  const int n_pairs = (n_tiles + 1) / 2;
  int splits = sm_count() / n_pairs;
  if (splits < 1) splits = 1;
  if (splits > n_stage_total) splits = n_stage_total;
  w.stages_per_split = (n_stage_total + splits - 1) / splits;
  splits = (n_stage_total + w.stages_per_split - 1) / w.stages_per_split;
  const W2Smem wl = w2_layout(L, Hp, F);
  DTB_CUDA_OK(cudaFuncSetAttribute(cin_tc2_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wl.total));
  cin_tc2_wgrad_kernel<<<dim3(n_pairs, splits), kW2Threads, wl.total, st>>>(w);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int cin_tc2_launch_fwd(const CinTcParams& p, int D, cudaStream_t st) {
  if (D == 16) return tc2_launch<16>(p, st);
  if (D == 32) return tc2_launch<32>(p, st);
  set_error("cin_tc2: embedding dim %d unsupported", D);
  return DTB_ERR_UNSUPPORTED;
}

}  // namespace dtb
