// tcgen05 / TMEM / TMA "tap GEMM" for sm_100a:
//   C[b][m][n] = epi( sum_{tap} sum_k A[b][m + shift[tap]][k] * W[n][tap*Kp + k] )
// A is a channels-last activation tensor [B][T][K] (bf16); rows outside [0,T) read as zero (TMA OOB fill), which
// is exactly the causal left padding of the reference's Conv1d (…tokenizer_v2.py:159-192) — no im2col buffer.
// A plain Linear is ntaps=1, shift=0; a causal ConvTranspose1d(k=2r, stride=r) is 2 taps with N = r*Cout.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

enum GemmAct { ACT_NONE = 0, ACT_SNAKE = 1, ACT_GELU = 2, ACT_SWIGLU_PAIR = 3, ACT_SWIGLU_BLK8 = 4 };

struct GemmEpilogue {
  const float* bias;      // [cmod] or null; channel = n % cmod
  const float* scale;     // [cmod] or null (LayerScale / ConvNeXt gamma), applied before the residual add
  const bf16* resid;      // [B][T][N] or null
  const float* snake_ea;  // exp(alpha) per channel (ACT_SNAKE)
  const float* snake_ib;  // 1/(exp(beta)+1e-9) per channel
  int cmod;               // channel modulus (Cout); N for plain layers
  int act;
  bf16* out_raw;          // [B][T][N] or null: value before the activation (residual stream)
  bf16* out_act;          // [B][T][N] (or [B][T][N/2] for ACT_SWIGLU_PAIR) or null
};

struct GemmPlan {
  CUtensorMap tmA, tmW;
  int B, T, N, Kp, ntaps, bn;
  int nst;                          // depth of the TMA ring (4, or 3 for the widest tiles: the epilogue staging needs 48 KB)
  int shift[8];
  int a_row0;                       // added to every A row coordinate (history-prefixed inputs of the streaming codec)
  long long raw_bs, act_bs, resid_bs;  // batch strides (elements) of out_raw / out_act / resid; rows are N (N/2) wide
  GemmEpilogue ep;
};

// Views for tensors that are not a plain contiguous [B][T][*]: the A map may cover more rows than the T output rows
// (a history prefix of a_row0 rows that the taps' negative shifts reach into), and every output / residual tensor
// may sit inside a larger per-batch allocation.  0 strides mean "contiguous".
struct GemmViews {
  int a_rows = 0;       // rows of the A map per batch (0 -> T)
  int a_row0 = 0;
  long long raw_bs = 0, act_bs = 0, resid_bs = 0;
};

// Encode the two tensor maps for a problem (host).  a: [B][T][K] bf16 with row pitch lda (elements) and batch
// stride (elements); w: [N][ntaps*Kp] bf16.  Returns 0 on success.
int gemm_make_plan(GemmPlan* plan, const bf16* a, int B, int T, int K, int64_t lda, int64_t a_batch_stride,
                   const bf16* w, int N, int Kp, int ntaps, const int* shifts, int bn, const GemmEpilogue& ep);
int gemm_make_plan_v(GemmPlan* plan, const bf16* a, int B, int T, int K, int64_t lda, int64_t a_batch_stride, const bf16* w,
                     int N, int Kp, int ntaps, const int* shifts, int bn, const GemmEpilogue& ep, const GemmViews& v);
// max_ctas > 0 caps the persistent grid below one CTA per SM (tests: more tiles per CTA on the same problem)
int gemm_launch(const GemmPlan& plan, cudaStream_t stream, int max_ctas = 0);
int gemm_init();  // resolves cuTensorMapEncodeTiled, sets kernel attributes
int gemm_pick_bn(int N, int mtiles, int B);  // largest tile width that still fills the 148 SMs
