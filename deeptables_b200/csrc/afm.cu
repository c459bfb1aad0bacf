// AFM -- attentional factorization machine (reference layers.py:742-812, afm_nets deepnets.py:99-107), gather fused.
//
//   v_p = e_i * e_j                    for the P = F(F-1)/2 field pairs (i < j, row-major = itertools.combinations)
//   a_p = act(v_p Wa + ba)             Dense(hidden_factor H), Wa [D, H]
//   s_p = a_p . h                      projection_h [H, 1];   w = softmax over the PAIRS of s
//   pooled[d] = sum_p w_p v_p[d]       [B, D]  -> Dropout -> Dense(1, no bias): those two are ordinary layers of this library
//
// 99 kFLOP per row against 1.7 KB of embedding rows: CUDA-core arithmetic out of shared memory, no tensor-core shape.
// Forward and the score half of the backward: one WARP per batch row, lanes = pairs (the softmax needs all pairs of a row).
// The per-pair backward writes da_p and dv_p = d v_p once per pair.  Embedding gradient: one THREAD per (row, field) -- it
// sums dv_p * e_other over the F-1 pairs of its field and keeps d e_f in registers (one vector RED per 4 floats at the end;
// every pair is read from both ends, which saves the scatter).  Attention-kernel gradient: warps stream (row, pair) outer
// products v_p (x) da_p into register accumulators, lane = (d, group of h).
// Widths are template parameters: DT = D in {4, 8, 16, 32}; HT = H rounded up to {8, 16, 32} with zero-padded columns
// (a padded unit has a = act(0) = 0 for relu / linear and h = 0, so it contributes nothing).
#include "dtb_common.cuh"

namespace dtb {

constexpr int kAfmWarps = 4;          // warps (= rows in flight) per CTA of the warp-per-row kernels; fewer when F is large (shared memory)
constexpr int kAfmRows = 128;         // rows (= threads) per CTA of the (row, field) kernel

// pairs (i < j) in row-major order = itertools.combinations (layers.py:794-796)
__device__ __forceinline__ void afm_pair_of(int p, int F, int& i, int& j) {
  int ii = 0, rem = p;
  while (rem >= F - 1 - ii) {
    rem -= F - 1 - ii;
    ++ii;
  }
  i = ii;
  j = ii + 1 + rem;
}
__device__ __forceinline__ int afm_pair_index(int a, int b, int F) { return a * (F - 1) - a * (a - 1) / 2 + (b - a - 1); }

__device__ __forceinline__ float afm_act(float x, int act) { return act == DTB_ACT_RELU ? fmaxf(x, 0.f) : x; }

template <int N>
__device__ __forceinline__ void afm_lds(const float* __restrict__ p, float (&o)[N]) {
#pragma unroll
  for (int c = 0; c < N / 4; ++c) {
    const float4 t = *reinterpret_cast<const float4*>(p + 4 * c);
    o[4 * c] = t.x;
    o[4 * c + 1] = t.y;
    o[4 * c + 2] = t.z;
    o[4 * c + 3] = t.w;
  }
}

// attention kernel / bias / projection into shared memory, columns padded to HT with zeros
template <int DT, int HT>
__device__ __forceinline__ void afm_stage_weights(const float* __restrict__ wa, const float* __restrict__ ba,
                                                  const float* __restrict__ hv, int H, float* __restrict__ s_wa,
                                                  float* __restrict__ s_ba, float* __restrict__ s_hv) {
  for (int e = threadIdx.x; e < DT * HT; e += blockDim.x) {
    const int d = e / HT, h = e - d * HT;
    s_wa[e] = h < H ? __ldg(wa + d * H + h) : 0.f;
  }
  for (int h = threadIdx.x; h < HT; h += blockDim.x) {
    s_ba[h] = h < H ? __ldg(ba + h) : 0.f;
    s_hv[h] = h < H ? __ldg(hv + h) : 0.f;
  }
}

// attention score of one pair: v = ei * ej (returned), a = act(v Wa + ba) (returned), s = a . h
template <int DT, int HT>
__device__ __forceinline__ float afm_score(const float (&ei)[DT], const float (&ej)[DT], const float* __restrict__ s_wa,
                                           const float* __restrict__ s_ba, const float* __restrict__ s_hv, int act,
                                           float (&a)[HT]) {
  afm_lds<HT>(s_ba, a);
#pragma unroll
  for (int d = 0; d < DT; ++d) {
    const float v = ei[d] * ej[d];
    float w[HT];
    afm_lds<HT>(s_wa + d * HT, w);
#pragma unroll
    for (int h = 0; h < HT; ++h) a[h] = fmaf(v, w[h], a[h]);
  }
  float hv[HT];
  afm_lds<HT>(s_hv, hv);
  float s = 0.f;
#pragma unroll
  for (int h = 0; h < HT; ++h) {
    a[h] = afm_act(a[h], act);
    s = fmaf(a[h], hv[h], s);
  }
  return s;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// shared memory of the warp-per-row kernels: [Wa DT*HT | ba HT | hv HT | pair table P (i | j << 16) |
//                                            per warp: es F*(DT+4) | sc P | dw P]
__host__ __device__ inline int afm_p4(int P) { return (P + 3) & ~3; }        // keeps every region 16-byte aligned
__host__ __device__ inline size_t afm_row_smem_floats(int F, int P, int DT, int HT, int n_warps) {
  return (size_t)DT * HT + 2 * HT + afm_p4(P) + (size_t)n_warps * ((size_t)F * (DT + 4) + 2 * (size_t)afm_p4(P));
}

// MODE 0: pooled[row, :] = sum_p softmax_p v_p.
// MODE 2: given g = dLoss/d pooled[row, :], the whole per-pair backward, each pair once: ds_p = w_p (g.v_p - sum_q w_q g.v_q),
//         da_p[h] = ds_p h[h] act'(a_p[h]) -> w_out [B, P, HT],
//         dv_p[d] = g[d] w_p + sum_h da_p[h] Wa[d][h] -> ds_out [B, P, DT], d h += ds_p a_p (afm_bwd_gather_kernel finishes).
template <int DT, int HT, int MODE>
__global__ void __launch_bounds__(kAfmWarps * 32) afm_rows_kernel(const int32_t* __restrict__ idx, const float* __restrict__ table,
                                                                  const int64_t* __restrict__ row_offsets,
                                                                  const float* __restrict__ wa, const float* __restrict__ ba,
                                                                  const float* __restrict__ hv, const float* __restrict__ g,
                                                                  float* __restrict__ pooled, float* __restrict__ w_out,
                                                                  float* __restrict__ ds_out, float* __restrict__ d_hv, int B,
                                                                  int F, int P, int H, int act, int* status) {
  constexpr bool BWD = MODE != 0;
  extern __shared__ __align__(16) float sm[];
  float* s_wa = sm;
  float* s_ba = s_wa + DT * HT;
  float* s_hv = s_ba + HT;
  uint32_t* s_pair = reinterpret_cast<uint32_t*>(s_hv + HT);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int RS = DT + 4;                                   // padded embedding row: conflict-free 128-bit reads
  const int P4 = afm_p4(P);
  float* es = reinterpret_cast<float*>(s_pair + P4) + (size_t)warp * ((size_t)F * RS + 2 * (size_t)P4);
  float* sc = es + (size_t)F * RS;
  float* dw = sc + P4;
  afm_stage_weights<DT, HT>(wa, ba, hv, H, s_wa, s_ba, s_hv);
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    int i, j;
    afm_pair_of(p, F, i, j);
    s_pair[p] = (uint32_t)i | ((uint32_t)j << 16);
  }
  __syncthreads();
  float dh_acc[HT];
#pragma unroll
  for (int h = 0; h < HT; ++h) dh_acc[h] = 0.f;
  const int n_warps = blockDim.x >> 5;         // kAfmWarps unless the host shrank the CTA to fit the shared memory
  for (int row = blockIdx.x * n_warps + warp; row < B; row += gridDim.x * n_warps) {
    __syncwarp();
    for (int e = lane; e < F * (DT / 4); e += 32) {
      const int f = e / (DT / 4), c = e - f * (DT / 4);
      const int64_t rb = table_row(row_offsets, f, __ldg(idx + (int64_t)row * F + f), DT, status);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (rb >= 0) v = __ldg(reinterpret_cast<const float4*>(table + rb) + c);
      *reinterpret_cast<float4*>(es + (size_t)f * RS + 4 * c) = v;
    }
    __syncwarp();
    float gr[DT];
    if (BWD) {
#pragma unroll
      for (int c = 0; c < DT / 4; ++c) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(g + (size_t)row * DT) + c);
        gr[4 * c] = t.x;
        gr[4 * c + 1] = t.y;
        gr[4 * c + 2] = t.z;
        gr[4 * c + 3] = t.w;
      }
    }
    float m = -INFINITY;
    for (int p = lane; p < P; p += 32) {
      const uint32_t ij = s_pair[p];
      float ei[DT], ej[DT], a[HT];
      afm_lds<DT>(es + (size_t)(ij & 0xffff) * RS, ei);
      afm_lds<DT>(es + (size_t)(ij >> 16) * RS, ej);
      const float s = afm_score<DT, HT>(ei, ej, s_wa, s_ba, s_hv, act, a);
      sc[p] = s;
      m = fmaxf(m, s);
      if (BWD) {
        float t = 0.f;
#pragma unroll
        for (int d = 0; d < DT; ++d) t = fmaf(gr[d], ei[d] * ej[d], t);
        dw[p] = t;
      }
    }
    m = warp_max(m);
    float sum = 0.f, dsum = 0.f, acc[DT];
#pragma unroll
    for (int d = 0; d < DT; ++d) acc[d] = 0.f;
    for (int p = lane; p < P; p += 32) {
      const float w = __expf(sc[p] - m);
      sum += w;
      if (BWD) {
        dsum = fmaf(w, dw[p], dsum);
        sc[p] = w;
      } else {
        const uint32_t ij = s_pair[p];
        float ei[DT], ej[DT];
        afm_lds<DT>(es + (size_t)(ij & 0xffff) * RS, ei);
        afm_lds<DT>(es + (size_t)(ij >> 16) * RS, ej);
#pragma unroll
        for (int d = 0; d < DT; ++d) acc[d] = fmaf(w, ei[d] * ej[d], acc[d]);
      }
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    if (MODE == 2) {
      const float delta = warp_sum(dsum) * inv;
      for (int p = lane; p < P; p += 32) {
        const float w = sc[p] * inv;
        const float ds = w * (dw[p] - delta);
        const uint32_t ij = s_pair[p];
        float a[HT];
        {
          float ei[DT], ej[DT];
          afm_lds<DT>(es + (size_t)(ij & 0xffff) * RS, ei);
          afm_lds<DT>(es + (size_t)(ij >> 16) * RS, ej);
          afm_score<DT, HT>(ei, ej, s_wa, s_ba, s_hv, act, a);
        }
        float hvr[HT];
        afm_lds<HT>(s_hv, hvr);
#pragma unroll
        for (int h = 0; h < HT; ++h) {
          dh_acc[h] = fmaf(ds, a[h], dh_acc[h]);
          const float slope = (act == DTB_ACT_RELU && !(a[h] > 0.f)) ? 0.f : 1.f;
          a[h] = ds * hvr[h] * slope;            // a[] now holds da
        }
        float4* da_dst = reinterpret_cast<float4*>(w_out + ((size_t)row * P + p) * HT);
#pragma unroll
        for (int c = 0; c < HT / 4; ++c) da_dst[c] = make_float4(a[4 * c], a[4 * c + 1], a[4 * c + 2], a[4 * c + 3]);
        float dv[DT];
#pragma unroll
        for (int d = 0; d < DT; ++d) {
          float wr[HT];
          afm_lds<HT>(s_wa + d * HT, wr);
          float t = gr[d] * w;
#pragma unroll
          for (int h = 0; h < HT; ++h) t = fmaf(a[h], wr[h], t);
          dv[d] = t;
        }
        float4* dv_dst = reinterpret_cast<float4*>(ds_out + ((size_t)row * P + p) * DT);
#pragma unroll
        for (int c = 0; c < DT / 4; ++c) dv_dst[c] = make_float4(dv[4 * c], dv[4 * c + 1], dv[4 * c + 2], dv[4 * c + 3]);
      }
    } else {
#pragma unroll
      for (int d = 0; d < DT; ++d) acc[d] = warp_sum(acc[d]);
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < DT / 4; ++c)
          reinterpret_cast<float4*>(pooled + (size_t)row * DT)[c] =
              make_float4(acc[4 * c] * inv, acc[4 * c + 1] * inv, acc[4 * c + 2] * inv, acc[4 * c + 3] * inv);
      }
    }
  }
  if (MODE == 2) {
#pragma unroll
    for (int h = 0; h < HT; ++h) {
      const float t = warp_sum(dh_acc[h]);
      if (lane == 0 && h < H && t != 0.f) atomicAdd(d_hv + h, t);
    }
  }
}

// d e_f = sum over the F-1 pairs that contain f of dv_p * e_other (dv_p from afm_rows_kernel<MODE 2>): thread = (row, field),
// grid (F, row-chunk groups); one vector RED per 4 floats.
template <int DT>
__global__ void __launch_bounds__(kAfmRows) afm_bwd_gather_kernel(const int32_t* __restrict__ idx, const float* __restrict__ table,
                                                                  const int64_t* __restrict__ row_offsets,
                                                                  const float* __restrict__ dv_in, float* __restrict__ grad_table,
                                                                  int B, int F, int P) {
  const int f = blockIdx.x;
  const int n_chunks = (B + kAfmRows - 1) / kAfmRows;
  for (int chunk = blockIdx.y; chunk < n_chunks; chunk += gridDim.y) {
    const int row = chunk * kAfmRows + threadIdx.x;
    if (row >= B) continue;
    const int64_t rb = table_row(row_offsets, f, __ldg(idx + (int64_t)row * F + f), DT, nullptr);
    if (rb < 0) continue;
    float acc[DT];
#pragma unroll
    for (int d = 0; d < DT; ++d) acc[d] = 0.f;
    for (int q = 0; q < F - 1; ++q) {
      const int o = q < f ? q : q + 1;
      const int p = o < f ? afm_pair_index(o, f, F) : afm_pair_index(f, o, F);
      const int64_t ro = table_row(row_offsets, o, __ldg(idx + (int64_t)row * F + o), DT, nullptr);
      if (ro < 0) continue;
      const float4* ev = reinterpret_cast<const float4*>(table + ro);
      const float4* dv = reinterpret_cast<const float4*>(dv_in + ((size_t)row * P + p) * DT);
#pragma unroll
      for (int c = 0; c < DT / 4; ++c) {
        const float4 e = __ldg(ev + c), t = __ldg(dv + c);
        acc[4 * c] = fmaf(t.x, e.x, acc[4 * c]);
        acc[4 * c + 1] = fmaf(t.y, e.y, acc[4 * c + 1]);
        acc[4 * c + 2] = fmaf(t.z, e.z, acc[4 * c + 2]);
        acc[4 * c + 3] = fmaf(t.w, e.w, acc[4 * c + 3]);
      }
    }
    float4* dst = reinterpret_cast<float4*>(grad_table + rb);
#pragma unroll
    for (int c = 0; c < DT / 4; ++c) {
      const float4 v = make_float4(acc[4 * c], acc[4 * c + 1], acc[4 * c + 2], acc[4 * c + 3]);
      if (v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f) atomicAdd(dst + c, v);
    }
  }
}

// d Wa[d][h] = sum_{row, p} v_p[d] da_p[h],  d ba[h] = sum da_p[h].  One warp streams rows; lane = (d, group of G = DT*HT/32 units).
template <int DT, int HT>
__global__ void __launch_bounds__(kAfmWarps * 32) afm_bwd_dw_kernel(const int32_t* __restrict__ idx, const float* __restrict__ table,
                                                                    const int64_t* __restrict__ row_offsets,
                                                                    const float* __restrict__ da_in, float* __restrict__ d_wa,
                                                                    float* __restrict__ d_ba, int B, int F, int P, int H) {
  constexpr int G = DT * HT / 32;               // units per lane (>= 1 for DT >= 4, HT >= 8)
  constexpr int RS = DT + 4;
  extern __shared__ __align__(16) float sm[];
  uint32_t* s_pair = reinterpret_cast<uint32_t*>(sm);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* es = reinterpret_cast<float*>(s_pair + afm_p4(P)) + (size_t)warp * ((size_t)F * RS + 32 * HT);
  float* das = es + (size_t)F * RS;             // [32 pairs][HT]
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    int i, j;
    afm_pair_of(p, F, i, j);
    s_pair[p] = (uint32_t)i | ((uint32_t)j << 16);
  }
  __syncthreads();
  const int d = lane % DT, h0 = (lane / DT) * G;
  float acc[G], accb[G];
#pragma unroll
  for (int k = 0; k < G; ++k) acc[k] = accb[k] = 0.f;
  const int n_warps = blockDim.x >> 5;         // kAfmWarps unless the host shrank the CTA to fit the shared memory
  for (int row = blockIdx.x * n_warps + warp; row < B; row += gridDim.x * n_warps) {
    __syncwarp();
    for (int e = lane; e < F * (DT / 4); e += 32) {
      const int f = e / (DT / 4), c = e - f * (DT / 4);
      const int64_t rb = table_row(row_offsets, f, __ldg(idx + (int64_t)row * F + f), DT, nullptr);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (rb >= 0) v = __ldg(reinterpret_cast<const float4*>(table + rb) + c);
      *reinterpret_cast<float4*>(es + (size_t)f * RS + 4 * c) = v;
    }
    for (int p0 = 0; p0 < P; p0 += 32) {
      __syncwarp();
      const int np = min(32, P - p0);
      // the chunk's da rows: np * HT contiguous floats, read as float4 by the whole warp
      const float4* src = reinterpret_cast<const float4*>(da_in + ((size_t)row * P + p0) * HT);
      for (int e = lane; e < np * (HT / 4); e += 32) reinterpret_cast<float4*>(das)[e] = __ldg(src + e);
      __syncwarp();
      for (int q = 0; q < np; ++q) {
        const uint32_t ij = s_pair[p0 + q];
        const float v = es[(size_t)(ij & 0xffff) * RS + d] * es[(size_t)(ij >> 16) * RS + d];
        float t[G];
        if constexpr (G % 4 == 0) {
          afm_lds<G>(das + q * HT + h0, t);
        } else {
#pragma unroll
          for (int k = 0; k < G; ++k) t[k] = das[q * HT + h0 + k];
        }
#pragma unroll
        for (int k = 0; k < G; ++k) {
          acc[k] = fmaf(v, t[k], acc[k]);
          if (d == 0) accb[k] += t[k];
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < G; ++k) {
    if (h0 + k < H) {
      if (acc[k] != 0.f) atomicAdd(d_wa + d * H + h0 + k, acc[k]);
      if (d == 0 && accb[k] != 0.f) atomicAdd(d_ba + h0 + k, accb[k]);
    }
  }
}

}  // namespace dtb

using namespace dtb;

namespace {
bool afm_shape(int D, int H, const void* table) {
  return (D == 4 || D == 8 || D == 16 || D == 32) && H >= 1 && H <= 32 && (reinterpret_cast<uintptr_t>(table) & 15) == 0;
}
int afm_ht(int H) { return H <= 8 ? 8 : (H <= 16 ? 16 : 32); }
constexpr size_t kAfmSmemMax = 200 * 1024;
}  // namespace

#define DTB_AFM_DISPATCH(D, HT, ...)                                                  \
  switch ((D) * 100 + (HT)) {                                                           \
    case 408: { constexpr int DT_ = 4, HT_ = 8; __VA_ARGS__; } break;                          \
    case 416: { constexpr int DT_ = 4, HT_ = 16; __VA_ARGS__; } break;                         \
    case 432: { constexpr int DT_ = 4, HT_ = 32; __VA_ARGS__; } break;                         \
    case 808: { constexpr int DT_ = 8, HT_ = 8; __VA_ARGS__; } break;                          \
    case 816: { constexpr int DT_ = 8, HT_ = 16; __VA_ARGS__; } break;                         \
    case 832: { constexpr int DT_ = 8, HT_ = 32; __VA_ARGS__; } break;                         \
    case 1608: { constexpr int DT_ = 16, HT_ = 8; __VA_ARGS__; } break;                        \
    case 1616: { constexpr int DT_ = 16, HT_ = 16; __VA_ARGS__; } break;                       \
    case 1632: { constexpr int DT_ = 16, HT_ = 32; __VA_ARGS__; } break;                       \
    case 3208: { constexpr int DT_ = 32, HT_ = 8; __VA_ARGS__; } break;                        \
    case 3216: { constexpr int DT_ = 32, HT_ = 16; __VA_ARGS__; } break;                       \
    case 3232: { constexpr int DT_ = 32, HT_ = 32; __VA_ARGS__; } break;                       \
    default: break;                                                                     \
  }

extern "C" {

size_t dtb_afm_workspace_bytes(int B, int F, int D, int H) {
  if (B <= 0 || F < 2 || H < 1 || H > 32 || D < 1) return 0;
  const size_t P = (size_t)F * (F - 1) / 2;
  const size_t per_pair = afm_ht(H) + (size_t)D;      // da + dv per pair
  return (size_t)B * P * per_pair * sizeof(float) + 256;
}

int dtb_afm_fwd(const int32_t* idx, const float* table, const int64_t* row_offsets, const float* att_kernel,
                const float* att_bias, const float* projection_h, float* pooled, int B, int F, int D, int H, int act,
                int* status, void* stream) {
  DTB_CHECK_ARG(idx && table && row_offsets && att_kernel && att_bias && projection_h && pooled, "NULL argument");
  DTB_CHECK_ARG(F >= 2 && F <= 4096 && B >= 0, "need 2 <= F <= 4096");
  DTB_CHECK_ARG(act == DTB_ACT_NONE || act == DTB_ACT_RELU, "attention activation must be linear or relu");
  if (!afm_shape(D, H, table) || (reinterpret_cast<uintptr_t>(pooled) & 15)) {
    set_error("dtb_afm_fwd: needs D in {4, 8, 16, 32}, hidden_factor <= 32 and 16-byte aligned buffers (D = %d, H = %d)", D, H);
    return DTB_ERR_UNSUPPORTED;
  }
  if (B == 0) return DTB_OK;
  const int P = F * (F - 1) / 2, HT = afm_ht(H);
  int nw = kAfmWarps;                            // many fields (an FGCNN block has ~100): fewer rows in flight per CTA
  while (nw > 1 && afm_row_smem_floats(F, P, D, HT, nw) * sizeof(float) > kAfmSmemMax) nw /= 2;
  const size_t smem = afm_row_smem_floats(F, P, D, HT, nw) * sizeof(float);
  if (smem > kAfmSmemMax) {
    set_error("dtb_afm_fwd: %d fields need %zu bytes of shared memory per CTA", F, smem);
    return DTB_ERR_UNSUPPORTED;
  }
  int grid = sm_count() * 4;
  if (grid > ceil_div(B, nw)) grid = ceil_div(B, nw);
  DTB_AFM_DISPATCH(D, HT, {
    auto kern = afm_rows_kernel<DT_, HT_, 0>;
    DTB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, nw * 32, smem, (cudaStream_t)stream>>>(idx, table, row_offsets, att_kernel, att_bias, projection_h,
                                                               nullptr, pooled, nullptr, nullptr, nullptr, B, F, P, H, act, status);
  })
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int dtb_afm_bwd(const int32_t* idx, const float* table, const int64_t* row_offsets, const float* att_kernel,
                const float* att_bias, const float* projection_h, const float* d_pooled, float* grad_table,
                float* d_att_kernel, float* d_att_bias, float* d_projection_h, void* workspace, size_t workspace_bytes,
                int B, int F, int D, int H, int act, void* stream) {
  DTB_CHECK_ARG(idx && table && row_offsets && att_kernel && att_bias && projection_h && d_pooled && grad_table &&
                    d_att_kernel && d_att_bias && d_projection_h,
                "NULL argument");
  DTB_CHECK_ARG(F >= 2 && F <= 4096 && B >= 0, "need 2 <= F <= 4096");
  DTB_CHECK_ARG(act == DTB_ACT_NONE || act == DTB_ACT_RELU, "attention activation must be linear or relu");
  if (!afm_shape(D, H, table) || ((reinterpret_cast<uintptr_t>(d_pooled) | reinterpret_cast<uintptr_t>(grad_table)) & 15)) {
    set_error("dtb_afm_bwd: needs D in {4, 8, 16, 32}, hidden_factor <= 32 and 16-byte aligned buffers (D = %d, H = %d)", D, H);
    return DTB_ERR_UNSUPPORTED;
  }
  if (B == 0) return DTB_OK;
  DTB_CHECK_ARG(workspace && workspace_bytes >= dtb_afm_workspace_bytes(B, F, D, H) &&
                    (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
                "workspace missing, misaligned or smaller than dtb_afm_workspace_bytes");
  const int P = F * (F - 1) / 2, HT = afm_ht(H);
  cudaStream_t st = (cudaStream_t)stream;
  int nw = kAfmWarps, nw_w = kAfmWarps;
  while (nw > 1 && afm_row_smem_floats(F, P, D, HT, nw) * sizeof(float) > kAfmSmemMax) nw /= 2;
  auto dw_smem = [&](int n) { return ((size_t)afm_p4(P) + (size_t)n * ((size_t)F * (D + 4) + 32 * HT)) * sizeof(float); };
  while (nw_w > 1 && dw_smem(nw_w) > kAfmSmemMax) nw_w /= 2;
  const size_t smem = afm_row_smem_floats(F, P, D, HT, nw) * sizeof(float);
  const size_t smem_w = dw_smem(nw_w);
  if (smem > kAfmSmemMax || smem_w > kAfmSmemMax) {
    set_error("dtb_afm_bwd: %d fields need %zu bytes of shared memory per CTA", F, smem > smem_w ? smem : smem_w);
    return DTB_ERR_UNSUPPORTED;
  }
  int grid = sm_count() * 4;
  if (grid > ceil_div(B, nw)) grid = ceil_div(B, nw);
  int g2 = ceil_div(sm_count() * 8, F);
  if (g2 > ceil_div(B, kAfmRows)) g2 = ceil_div(B, kAfmRows);
  int grid_w = sm_count() * 2;
  if (grid_w > ceil_div(B, nw_w)) grid_w = ceil_div(B, nw_w);
  float* da = reinterpret_cast<float*>(workspace);              // da [B, P, HT] | dv [B, P, D]
  float* dv = da + (size_t)B * P * HT;
  DTB_AFM_DISPATCH(D, HT, {
    auto k1 = afm_rows_kernel<DT_, HT_, 2>;
    DTB_CUDA_OK(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k1<<<grid, nw * 32, smem, st>>>(idx, table, row_offsets, att_kernel, att_bias, projection_h, d_pooled, nullptr, da, dv,
                                    d_projection_h, B, F, P, H, act, nullptr);
    afm_bwd_gather_kernel<DT_><<<dim3(F, g2), kAfmRows, 0, st>>>(idx, table, row_offsets, dv, grad_table, B, F, P);
    auto k3 = afm_bwd_dw_kernel<DT_, HT_>;
    DTB_CUDA_OK(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));
    k3<<<grid_w, nw_w * 32, smem_w, st>>>(idx, table, row_offsets, da, d_att_kernel, d_att_bias, B, F, P, H);
  })
  DTB_LAUNCH_OK();
  return DTB_OK;
}

}  // extern "C"
