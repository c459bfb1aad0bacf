// Definitions shared by the two translation units of the tensor-core CIN: cin_tc.cu (bf16x3 kernels for every
// supported shape, host side) and cin_tc2.cu (the restructured single-pass fp16 kernels).
#pragma once
#include "dtb_common.cuh"
#include "cin_shapes.h"
#include "tcgen05.cuh"

namespace dtb {

constexpr int kMaxL = 128;      // feature maps per layer (UMMA N)
constexpr int kMaxHp = 64;      // padded hidden fields per layer (K chunk)
constexpr int kTcThreads = 320;
constexpr int kAccCols = 128;   // TMEM columns per accumulator tile
constexpr int kTmemCols = 512;

struct CinTcParams {
  const int32_t* idx;
  const float* table;
  const int64_t* row_offsets;
  const uint8_t* wpack;
  const float* bias;
  float* pooled;
  float* saved;       // training: x0t [B,D,F] then T_k [B,D,L_k] (same layout as the fp32 path)
  int* status;
  int B, F, n_layers, act, n_pass, P;
  int L[kCinMaxLayers], H[kCinMaxLayers], Hp[kCinMaxLayers];
  int pool_lo[kCinMaxLayers], pool_n[kCinMaxLayers], pcol0[kCinMaxLayers], hid_n[kCinMaxLayers];
  unsigned long long wpack_off[kCinMaxLayers];   // byte offset of layer k's chunk images
  unsigned long long saved_off[kCinMaxLayers];   // float offset of T_k inside saved
  unsigned long long hb_off[kCinMaxLayers];      // float offset of the block-transposed copy of h_{k+1} = T_k[:, :hid_n]
  unsigned long long xb_off;                     // float offset of the block-transposed copy of x0
  unsigned long long bias_off[kCinMaxLayers];
  int b_stage_bytes;                              // bytes reserved per weight stage in smem
  int compact;                                    // training: save relu-mask bits instead of the fp32 T_k rows (see cin_tc_compact)
  const int* wmax;                                // cin_tc2: bit pattern of max|W_k| per layer (cin_tc_wmax_kernel)
};

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

constexpr int kSubK = 32;
constexpr int kStagesA = 4;
constexpr int kStagesB = 4;
constexpr int kACols = kSubK / 2;                 // TMEM columns of one bf16 [128 x 32] operand block
constexpr int kWgPad = 68;                        // row stride (floats) of the block-transposed tiles the wgrad kernel reads

__device__ __forceinline__ bool elect_one_sync() {
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

struct CinTcBwdParams {
  const int32_t* idx;
  const float* table;
  const int64_t* row_offsets;
  const uint8_t* wpack;       // transposed pack (B[n=j][k=l])
  const float* d_pooled;
  const float* saved;
  float* grad_table;
  uint8_t* dc_tiles;
  int B, F, n_layers, act, n_pass, P;
  int L[kCinMaxLayers], H[kCinMaxLayers], Hp[kCinMaxLayers];
  int pool_lo[kCinMaxLayers], pool_n[kCinMaxLayers], pcol0[kCinMaxLayers], hid_n[kCinMaxLayers];
  unsigned long long wpack_off[kCinMaxLayers], saved_off[kCinMaxLayers], dc_off[kCinMaxLayers];
  unsigned long long hb_off[kCinMaxLayers];      // float offset of the block-transposed h_{k+1} tiles (as in CinTcParams)
  int b_stage_bytes;
  int compact;                                    // saved activations in the compact format (cin_tc_compact)
  const int* wmax;                                // cin_tc2: statistics words (max|W_k| per layer at [k], max|dC_k| at [8 + k])
  const float* dpmax;                             // cin_tc2: max|d_pooled[b, pooled columns of layer k]|, [B, n_layers]
};


// ---- cin_tc2.cu: single-pass fp16 kernels with two threads per GEMM row (see the file header) -------------------------
bool cin_tc2_fwd_supported(const CinTcParams& p, int D);
int cin_tc2_launch_fwd(const CinTcParams& p, int D, cudaStream_t st);
bool cin_tc2_bwd_supported(const CinTcBwdParams& p, int D);
int cin_tc2_launch_dgrad(const CinTcBwdParams& p, int D, cudaStream_t st);
int cin_tc2_dpmax(const float* d_pooled, float* out, const int* pcol0_host, const int* pool_n_host, int B, int P, int n_layers,
                  cudaStream_t st);
int cin_tc2_dbias(const uint8_t* dc_tiles, float* d_bias, int L, int n_blocks16, cudaStream_t st);
bool cin_tc2_wgrad_supported(int F, int Hp, int L);
int cin_tc2_launch_wgrad(const float* xb, const float* hb, const uint8_t* dc_tiles, float* d_w, int F, int H, int Hp, int L,
                         int n_stage_total, const int* stats, int layer, cudaStream_t st);

}  // namespace dtb
