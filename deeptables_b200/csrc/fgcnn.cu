// FGCNN feature generation (reference layers.py:161-242; fg_nets deepnets.py:227-261): per layer
//   Conv2D(filters, kernel_size = (kh, 1), 'same', activation) along the FIELD axis of a channels-last block X [B, H, W, Cin]
//   (H = fields, W = embedding width), MaxPooling2D((pool, 1), 'same') along the same axis, then Flatten + Dense (a Dense call
//   of this library with the tanh epilogue) that recombines the pooled maps into new fields.
// Both ops are 1-D along H with the (W, C) plane riding along: a thread owns one (b, h, w) position and all its channels.
// The convolution is a [positions x (kh Cin)] x [(kh Cin) x Cout] product with Cout <= 32 and kh Cin <= 8 * 32: CUDA-core FMAs
// with the filter in shared memory (read as 128-bit warp broadcasts) -- 43 GFLOP per 65 536-row step at the reference's
// defaults (14 / 16 filters, height 7) against 1.5 GB of activations, i.e. bandwidth and issue bound, not a tensor-core shape.
#include "dtb_common.cuh"

namespace dtb {

constexpr int kFgThreads = 256;
constexpr int kFgMaxKh = 8;

// TensorFlow 'SAME' padding in front of an axis (the remainder goes behind): total = max((out-1) stride + k - size, 0)
__host__ __device__ inline int fg_pad_before(int size, int k, int stride) {
  const int out = (size + stride - 1) / stride;
  int total = (out - 1) * stride + k - size;
  if (total < 0) total = 0;
  return total / 2;
}

__device__ __forceinline__ float fg_act(float v, int act) {
  return act == DTB_ACT_RELU ? fmaxf(v, 0.f) : (act == DTB_ACT_TANH ? tanhf(v) : v);
}
// derivative of the activation expressed with its OUTPUT y
__device__ __forceinline__ float fg_act_grad(float y, int act) {
  return act == DTB_ACT_RELU ? (y > 0.f ? 1.f : 0.f) : (act == DTB_ACT_TANH ? 1.f - y * y : 1.f);
}

// Y[b,h,w,co] = act(bias[co] + sum_{t,ci} X[b, h + t - pad, w, ci] K[t, ci, co]).  CP = Cout rounded up to 8 / 16 / 32.
template <int CP>
__global__ void __launch_bounds__(kFgThreads) conv_fields_fwd_kernel(const float* __restrict__ X, const float* __restrict__ K,
                                                                     const float* __restrict__ bias, float* __restrict__ Y,
                                                                     int64_t n_pos, int H, int W, int Cin, int Cout, int kh,
                                                                     int act) {
  extern __shared__ __align__(16) float sk[];            // [kh][Cin][CP] | bias [CP]
  float* sb = sk + (size_t)kh * Cin * CP;
  for (int e = threadIdx.x; e < kh * Cin * CP; e += blockDim.x) {
    const int co = e % CP, r = e / CP;
    sk[e] = co < Cout ? __ldg(K + (size_t)r * Cout + co) : 0.f;
  }
  for (int co = threadIdx.x; co < CP; co += blockDim.x) sb[co] = (co < Cout && bias) ? __ldg(bias + co) : 0.f;
  __syncthreads();
  const int pad = fg_pad_before(H, kh, 1);
  for (int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pos < n_pos; pos += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(pos % W);
    const int64_t bh = pos / W;
    const int h = (int)(bh % H);
    float acc[CP];
#pragma unroll
    for (int c = 0; c < CP / 4; ++c) {
      const float4 t = *reinterpret_cast<const float4*>(sb + 4 * c);
      acc[4 * c] = t.x; acc[4 * c + 1] = t.y; acc[4 * c + 2] = t.z; acc[4 * c + 3] = t.w;
    }
    for (int t = 0; t < kh; ++t) {
      const int hh = h + t - pad;
      if (hh < 0 || hh >= H) continue;
      const float* xp = X + ((bh - h + hh) * W + w) * Cin;
      const float* kt = sk + (size_t)t * Cin * CP;
      for (int ci = 0; ci < Cin; ++ci) {
        const float x = __ldg(xp + ci);
#pragma unroll
        for (int c = 0; c < CP / 4; ++c) {
          const float4 k4 = *reinterpret_cast<const float4*>(kt + ci * CP + 4 * c);
          acc[4 * c] = fmaf(x, k4.x, acc[4 * c]);
          acc[4 * c + 1] = fmaf(x, k4.y, acc[4 * c + 1]);
          acc[4 * c + 2] = fmaf(x, k4.z, acc[4 * c + 2]);
          acc[4 * c + 3] = fmaf(x, k4.w, acc[4 * c + 3]);
        }
      }
    }
    float* y = Y + pos * Cout;
#pragma unroll
    for (int co = 0; co < CP; ++co)
      if (co < Cout) y[co] = fg_act(acc[co], act);
  }
}

// dX[b,h,w,ci] = sum_{t,co} dZ[b, h - t + pad, w, co] K[t, ci, co],  dZ = dY act'(Y).  CP = Cin rounded up to 8 / 16 / 32;
// the filter sits transposed in shared memory: [kh][Cout][CP].
template <int CP>
__global__ void __launch_bounds__(kFgThreads) conv_fields_bwd_dx_kernel(const float* __restrict__ Y, const float* __restrict__ dY,
                                                                        const float* __restrict__ K, float* __restrict__ dX,
                                                                        int64_t n_pos, int H, int W, int Cin, int Cout, int kh,
                                                                        int act) {
  extern __shared__ __align__(16) float sk[];            // [kh][Cout][CP]
  for (int e = threadIdx.x; e < kh * Cout * CP; e += blockDim.x) {
    const int ci = e % CP, r = e / CP, co = r % Cout, t = r / Cout;
    sk[e] = ci < Cin ? __ldg(K + ((size_t)t * Cin + ci) * Cout + co) : 0.f;
  }
  __syncthreads();
  const int pad = fg_pad_before(H, kh, 1);
  for (int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pos < n_pos; pos += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(pos % W);
    const int64_t bh = pos / W;
    const int h = (int)(bh % H);
    float acc[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) acc[c] = 0.f;
    for (int t = 0; t < kh; ++t) {
      const int hh = h - t + pad;                        // the output position whose tap t reads this input position
      if (hh < 0 || hh >= H) continue;
      const int64_t o = ((bh - h + hh) * W + w) * Cout;
      const float* kt = sk + (size_t)t * Cout * CP;
      for (int co = 0; co < Cout; ++co) {
        const float dz = __ldg(dY + o + co) * fg_act_grad(__ldg(Y + o + co), act);
#pragma unroll
        for (int c = 0; c < CP / 4; ++c) {
          const float4 k4 = *reinterpret_cast<const float4*>(kt + co * CP + 4 * c);
          acc[4 * c] = fmaf(dz, k4.x, acc[4 * c]);
          acc[4 * c + 1] = fmaf(dz, k4.y, acc[4 * c + 1]);
          acc[4 * c + 2] = fmaf(dz, k4.z, acc[4 * c + 2]);
          acc[4 * c + 3] = fmaf(dz, k4.w, acc[4 * c + 3]);
        }
      }
    }
    float* dx = dX + pos * Cin;
#pragma unroll
    for (int ci = 0; ci < CP; ++ci)
      if (ci < Cin) dx[ci] = acc[ci];
  }
}

// dK[t,ci,co] += sum_pos X[b, h + t - pad, w, ci] dZ[b,h,w,co];  dbias[co] += sum_pos dZ.  A CTA takes tiles of kFgTile
// consecutive positions, stages their taps xs[p][a] (a = t Cin + ci, zero outside the block) and dzs[p][co] in shared
// memory, and every thread accumulates its (a, co) entries -- dK is exactly the [A x Cout] matrix xs^T dzs in memory order --
// over the tile; accumulators live in registers across the CTA's tiles, one atomic per entry per CTA at the end.  (A first
// version that walked the positions serially with one (ci, co) entry per thread took 106 ms per launch at 65 536 rows.)
constexpr int kFgTile = 128;
constexpr int kFgMaxEntries = 32;        // (kh Cin Cout) / 256 threads, kh <= 8, Cin, Cout <= 32

__global__ void __launch_bounds__(kFgThreads) conv_fields_bwd_dw_tiled_kernel(const float* __restrict__ X, const float* __restrict__ Y,
                                                                              const float* __restrict__ dY, float* __restrict__ dK,
                                                                              float* __restrict__ dbias, int64_t n_pos, int H, int W,
                                                                              int Cin, int Cout, int kh, int act, int64_t n_tiles) {
  extern __shared__ __align__(16) float sm[];
  const int A = kh * Cin;
  float* xs = sm;                        // [kFgTile][A]
  float* dzs = sm + (size_t)kFgTile * A; // [kFgTile][Cout]
  const int n_out = A * Cout;
  const int pad = fg_pad_before(H, kh, 1);
  float acc[kFgMaxEntries];
#pragma unroll
  for (int k = 0; k < kFgMaxEntries; ++k) acc[k] = 0.f;
  float accb = 0.f;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t p0 = tile * kFgTile;
    __syncthreads();
    for (int i = threadIdx.x; i < kFgTile * A; i += kFgThreads) {
      const int p = i / A, a = i - p * A;
      const int64_t pos = p0 + p;
      float v = 0.f;
      if (pos < n_pos) {
        const int w = (int)(pos % W);
        const int64_t bh = pos / W;
        const int h = (int)(bh % H);
        const int t = a / Cin, ci = a - t * Cin;
        const int hh = h + t - pad;
        if (hh >= 0 && hh < H) v = __ldg(X + ((bh - h + hh) * W + w) * Cin + ci);
      }
      xs[i] = v;
    }
    for (int i = threadIdx.x; i < kFgTile * Cout; i += kFgThreads) {
      const int64_t pos = p0 + i / Cout;
      float v = 0.f;
      if (pos < n_pos) {
        const int64_t o = p0 * Cout + i;
        v = __ldg(dY + o) * fg_act_grad(__ldg(Y + o), act);
      }
      dzs[i] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kFgMaxEntries; ++k) {
      const int e = threadIdx.x + k * kFgThreads;
      if (e < n_out) {
        const int a = e / Cout, co = e - a * Cout;
        float s = 0.f;
        for (int p = 0; p < kFgTile; ++p) s = fmaf(xs[p * A + a], dzs[p * Cout + co], s);
        acc[k] += s;
      }
    }
    if (threadIdx.x < Cout) {
      float s = 0.f;
      for (int p = 0; p < kFgTile; ++p) s += dzs[p * Cout + threadIdx.x];
      accb += s;
    }
  }
#pragma unroll
  for (int k = 0; k < kFgMaxEntries; ++k) {
    const int e = threadIdx.x + k * kFgThreads;
    if (e < n_out && acc[k] != 0.f) atomicAdd(dK + e, acc[k]);
  }
  if (threadIdx.x < Cout && dbias && accb != 0.f) atomicAdd(dbias + threadIdx.x, accb);
}

// MaxPooling2D((pool, 1), strides = pool, 'same'): Y[b,ho,w,c] = max over the window's in-range rows; thread = output element
__global__ void maxpool_fields_fwd_kernel(const float* __restrict__ X, float* __restrict__ Y, int64_t n_out, int H, int Ho,
                                          int WC, int pool) {
  const int pad = fg_pad_before(H, pool, pool);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (int64_t)gridDim.x * blockDim.x) {
    const int wc = (int)(i % WC);
    const int64_t bo = i / WC;
    const int ho = (int)(bo % Ho);
    const int64_t b = bo / Ho;
    float m = -INFINITY;
    for (int k = 0; k < pool; ++k) {
      const int h = ho * pool - pad + k;
      if (h >= 0 && h < H) m = fmaxf(m, __ldg(X + (b * H + h) * WC + wc));
    }
    Y[i] = m;
  }
}
// the windows do not overlap (stride = pool): each output element writes the gradient of its own window, the first maximum
// takes it (TensorFlow's MaxPoolGrad / torch.max)
__global__ void maxpool_fields_bwd_kernel(const float* __restrict__ X, const float* __restrict__ dY, float* __restrict__ dX,
                                          int64_t n_out, int H, int Ho, int WC, int pool) {
  const int pad = fg_pad_before(H, pool, pool);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (int64_t)gridDim.x * blockDim.x) {
    const int wc = (int)(i % WC);
    const int64_t bo = i / WC;
    const int ho = (int)(bo % Ho);
    const int64_t b = bo / Ho;
    float m = -INFINITY;
    int arg = -1;
    for (int k = 0; k < pool; ++k) {
      const int h = ho * pool - pad + k;
      if (h < 0 || h >= H) continue;
      const float v = __ldg(X + (b * H + h) * WC + wc);
      if (arg < 0 || v > m) {
        m = v;
        arg = h;
      }
    }
    const float g = __ldg(dY + i);
    for (int k = 0; k < pool; ++k) {
      const int h = ho * pool - pad + k;
      if (h >= 0 && h < H) dX[(b * H + h) * WC + wc] = h == arg ? g : 0.f;
    }
  }
}

}  // namespace dtb

using namespace dtb;

namespace {
int fg_cp(int c) { return c <= 8 ? 8 : (c <= 16 ? 16 : 32); }
int fg_grid(int64_t n) {
  int64_t g = (n + kFgThreads - 1) / kFgThreads;
  const int64_t cap = (int64_t)sm_count() * 8;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}
}  // namespace

#define DTB_FG_DISPATCH(CPV, ...)                          \
  switch (CPV) {                                           \
    case 8: { constexpr int CP_ = 8; __VA_ARGS__; } break;   \
    case 16: { constexpr int CP_ = 16; __VA_ARGS__; } break; \
    case 32: { constexpr int CP_ = 32; __VA_ARGS__; } break; \
    default: break;                                        \
  }

extern "C" {

int dtb_conv_fields_fwd(const float* X, const float* kernel, const float* bias, float* Y, int B, int H, int W, int Cin, int Cout,
                        int kh, int act, void* stream) {
  DTB_CHECK_ARG(X && kernel && Y, "NULL argument");
  DTB_CHECK_ARG(B >= 0 && H >= 1 && W >= 1, "bad shape");
  DTB_CHECK_ARG(act == DTB_ACT_NONE || act == DTB_ACT_RELU || act == DTB_ACT_TANH, "unsupported activation");
  if (Cin < 1 || Cin > 32 || Cout < 1 || Cout > 32 || kh < 1 || kh > kFgMaxKh) {
    set_error("dtb_conv_fields_fwd: needs 1 <= channels, filters <= 32 and kernel height <= %d (Cin %d, Cout %d, kh %d)", kFgMaxKh,
              Cin, Cout, kh);
    return DTB_ERR_UNSUPPORTED;
  }
  const int64_t n_pos = (int64_t)B * H * W;
  if (n_pos == 0) return DTB_OK;
  const int cp = fg_cp(Cout);
  const size_t smem = ((size_t)kh * Cin * cp + cp) * sizeof(float);
  DTB_FG_DISPATCH(cp, {
    auto k = conv_fields_fwd_kernel<CP_>;
    DTB_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<fg_grid(n_pos), kFgThreads, smem, (cudaStream_t)stream>>>(X, kernel, bias, Y, n_pos, H, W, Cin, Cout, kh, act);
  })
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int dtb_conv_fields_bwd(const float* X, const float* kernel, const float* Y, const float* dY, float* dX, float* d_kernel,
                        float* d_bias, int B, int H, int W, int Cin, int Cout, int kh, int act, void* stream) {
  DTB_CHECK_ARG(X && kernel && Y && dY && d_kernel, "NULL argument");
  DTB_CHECK_ARG(B >= 0 && H >= 1 && W >= 1, "bad shape");
  DTB_CHECK_ARG(act == DTB_ACT_NONE || act == DTB_ACT_RELU || act == DTB_ACT_TANH, "unsupported activation");
  if (Cin < 1 || Cin > 32 || Cout < 1 || Cout > 32 || kh < 1 || kh > kFgMaxKh) {
    set_error("dtb_conv_fields_bwd: needs 1 <= channels, filters <= 32 and kernel height <= %d (Cin %d, Cout %d, kh %d)", kFgMaxKh,
              Cin, Cout, kh);
    return DTB_ERR_UNSUPPORTED;
  }
  const int64_t n_pos = (int64_t)B * H * W;
  if (n_pos == 0) return DTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dX) {
    const int cp = fg_cp(Cin);
    const size_t smem = (size_t)kh * Cout * cp * sizeof(float);
    DTB_FG_DISPATCH(cp, {
      auto k = conv_fields_bwd_dx_kernel<CP_>;
      DTB_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k<<<fg_grid(n_pos), kFgThreads, smem, st>>>(Y, dY, kernel, dX, n_pos, H, W, Cin, Cout, kh, act);
    })
    DTB_LAUNCH_OK();
  }
  const int64_t n_tiles = (n_pos + kFgTile - 1) / kFgTile;
  const size_t smem = (size_t)kFgTile * (kh * Cin + Cout) * sizeof(float);
  int64_t ctas = (int64_t)sm_count() * 2;
  if (ctas > n_tiles) ctas = n_tiles;
  DTB_CUDA_OK(cudaFuncSetAttribute(conv_fields_bwd_dw_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  conv_fields_bwd_dw_tiled_kernel<<<(int)ctas, kFgThreads, smem, st>>>(X, Y, dY, d_kernel, d_bias, n_pos, H, W, Cin, Cout, kh, act,
                                                                       n_tiles);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int dtb_maxpool_fields_fwd(const float* X, float* Y, int B, int H, int WC, int pool, void* stream) {
  DTB_CHECK_ARG(X && Y && B >= 0 && H >= 1 && WC >= 1 && pool >= 1, "bad argument");
  const int Ho = (H + pool - 1) / pool;
  const int64_t n = (int64_t)B * Ho * WC;
  if (n == 0) return DTB_OK;
  maxpool_fields_fwd_kernel<<<fg_grid(n), kFgThreads, 0, (cudaStream_t)stream>>>(X, Y, n, H, Ho, WC, pool);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

int dtb_maxpool_fields_bwd(const float* X, const float* dY, float* dX, int B, int H, int WC, int pool, void* stream) {
  DTB_CHECK_ARG(X && dY && dX && B >= 0 && H >= 1 && WC >= 1 && pool >= 1, "bad argument");
  const int Ho = (H + pool - 1) / pool;
  const int64_t n = (int64_t)B * Ho * WC;
  if (n == 0) return DTB_OK;
  maxpool_fields_bwd_kernel<<<fg_grid(n), kFgThreads, 0, (cudaStream_t)stream>>>(X, dY, dX, n, H, Ho, WC, pool);
  DTB_LAUNCH_OK();
  return DTB_OK;
}

}  // extern "C"
