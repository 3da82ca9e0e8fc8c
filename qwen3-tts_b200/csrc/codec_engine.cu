// Qwen3-TTS-Tokenizer-12Hz codec DECODER on B200 (sm_100a): codes -> 24 kHz waveform.
// Replaces Qwen3TTSTokenizerV2Decoder.forward (qwen_tts/core/tokenizer_12hz/modeling_qwen3_tts_tokenizer_v2.py:869-884).
//
// Layout: every activation is channels-last bf16 [B][T][C]; every Conv1d / ConvTranspose1d / Linear is ONE
// tcgen05 tap-GEMM launch (gemm_sm100.cu) whose A tiles are TMA-loaded with a per-tap row shift — no im2col
// buffer — with bias, LayerScale, residual add and the *next* layer's SnakeBeta fused into the epilogue.
// Small row-wise ops (RVQ gather, RMSNorm, RoPE, 72-frame sliding-window attention, depthwise conv + LayerNorm,
// the final 96->1 conv + clamp) are plain CUDA kernels: they are <2 % of the FLOPs and HBM-trivial.
#include "common.cuh"
#include "gemm_sm100.cuh"
#include "../../include/qwen3tts_b200.h"

#include <algorithm>
#include <map>
#include <string>
#include <vector>

namespace {

struct DevTensor {
  void* p = nullptr;
  int dtype = 0;  // 0 = bf16, 1 = f32
  int64_t numel = 0;
};

// ---------------------------------------------------------------------------------------------- small kernels
// RVQ decode (…v2.py:815-821, :721-727, :676-679): e[b][t][0:D] = table[0][c0]; e[b][t][D:2D] = sum_{k>=1} table[k][c_k]
__global__ void rvq_gather_kernel(const int* __restrict__ codes, const bf16* __restrict__ table, bf16* __restrict__ e,
                                  int B, int K, int T, int D, int bins) {
  const int bt = blockIdx.x;  // b*T + t
  const int b = bt / T, t = bt % T;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const int c0 = codes[((size_t)b * K + 0) * T + t];
    e[(size_t)bt * 2 * D + d] = table[((size_t)0 * bins + c0) * D + d];
    float acc = 0.f;
    for (int k = 1; k < K; ++k) {
      const int c = codes[((size_t)b * K + k) * T + t];
      const float v = bf2f(table[((size_t)k * bins + c) * D + d]);
      acc = (k == 1) ? v : rbf(acc + v);  // the reference accumulates in the model dtype
    }
    e[(size_t)bt * 2 * D + D + d] = f2bf(acc);
  }
}

// RMSNorm over the last dim (…v2.py:383-388): one warp per row
__global__ void rmsnorm_rows_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w, bf16* __restrict__ y, int rows,
                                    int C, float eps) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const bf16* xr = x + (size_t)row * C;
  float ss = 0.f;
  for (int i = lane; i < C; i += 32) { const float v = bf2f(xr[i]); ss += v * v; }
  ss = warp_sum(ss);
  const float inv = rsqrtf(ss / (float)C + eps);
  for (int i = lane; i < C; i += 32) y[(size_t)row * C + i] = f2bf(rbf(bf2f(xr[i]) * inv) * bf2f(w[i]));
}

// RoPE in place on the q and k heads of qkv [B][n][3*nh*hd] at positions pos0 + t (…v2.py:329, apply_rotary_pos_emb).
// Given a window buffer kv [B][kv_bs_rows][2*nh*hd] (streaming decoder), the rotated k heads and the v heads of the n
// rows are also appended to it at rows [hist, hist + n): [K heads | V heads].
__global__ void rope_kernel(bf16* __restrict__ qkv, const bf16* __restrict__ cosT, const bf16* __restrict__ sinT,
                            bf16* __restrict__ kv, int hist, int kv_bs_rows, int B, int n, int nh, int hd, int pos0) {
  const int half = hd / 2;
  const int heads = kv ? 3 * nh : 2 * nh;  // q heads, k heads (, v heads)
  const size_t total = (size_t)B * n * heads * half;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int f = (int)(i % half);
    const int h = (int)((i / half) % heads);
    const size_t bt = i / ((size_t)half * heads);
    const int t = (int)(bt % n);
    bf16* v = qkv + bt * (size_t)(3 * nh * hd) + (size_t)h * hd;
    if (h < 2 * nh) {
      const float c = bf2f(cosT[(size_t)(pos0 + t) * half + f]), s = bf2f(sinT[(size_t)(pos0 + t) * half + f]);
      const float x1 = bf2f(v[f]), x2 = bf2f(v[f + half]);
      v[f] = f2bf(rbf(x1 * c) + rbf(-x2 * s));
      v[f + half] = f2bf(rbf(x2 * c) + rbf(x1 * s));
    }
    if (kv && h >= nh) {
      bf16* d = kv + ((bt / n) * kv_bs_rows + hist + t) * (size_t)(2 * nh * hd) + (size_t)(h - nh) * hd;
      d[f] = v[f];
      d[f + half] = v[f + half];
    }
  }
}

// causal sliding-window attention of the n queries of qkv [B][n][3*nh*hd], one warp per (b, head, t) (…v2.py:321-354;
// window: key k visible iff 0 <= t-k < W).  Keys and values are rows of kv [B][kv_bs_rows][ld] (K heads from column 0,
// V heads from column nh*hd); row r holds absolute position pos0 - hist + r (rows of negative position are not valid
// yet) and query t is row hist + t.  One-shot: kv is the k part of qkv itself (ld = 3*nh*hd), hist = pos0 = 0.
__global__ void window_attention_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ kv, int ld, int kv_bs_rows,
                                        int hist, int pos0, bf16* __restrict__ out, int B, int n, int nh, int hd, int window) {
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (wid >= B * n * nh) return;
  const int lane = threadIdx.x & 31;
  const int h = wid % nh, t = (wid / nh) % n, b = wid / (nh * n);
  const bf16* q = qkv + ((size_t)b * n + t) * (size_t)(3 * nh * hd) + (size_t)h * hd;
  const int r1 = hist + t;                                   // the query's own row
  const int r0 = max(max(r1 - window + 1, hist - pos0), 0);  // oldest visible row
  const int nk = r1 - r0 + 1;
  const bf16* base = kv + (size_t)b * kv_bs_rows * ld;
  const float scale = rsqrtf((float)hd);
  // scores: lane handles keys lane, lane+32, lane+64 (window <= 96)
  float sc[3];
  float mx = -INFINITY;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int kk = lane + 32 * r;
    sc[r] = -INFINITY;
    if (kk < nk) {
      const bf16* kp = base + (size_t)(r0 + kk) * ld + (size_t)h * hd;
      float d = 0.f;
      for (int i = 0; i < hd; i += 2) {
        const uint32_t qa = *reinterpret_cast<const uint32_t*>(q + i), ka = *reinterpret_cast<const uint32_t*>(kp + i);
        d += bf16lo(qa) * bf16lo(ka) + bf16hi(qa) * bf16hi(ka);
      }
      sc[r] = rbf(rbf(d) * scale);  // bf16 matmul output, then * scaling in bf16 (eager path)
      mx = fmaxf(mx, sc[r]);
    }
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int r = 0; r < 3; ++r) { sc[r] = (sc[r] == -INFINITY) ? 0.f : __expf(sc[r] - mx); sum += sc[r]; }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  // output: lanes over dims (hd <= 64 -> 2 per lane), loop over keys with shuffles
  float o0 = 0.f, o1 = 0.f;
  for (int kk = 0; kk < nk; ++kk) {
    const float p = rbf(__shfl_sync(0xffffffffu, sc[kk >> 5], kk & 31) * inv);  // softmax cast to bf16
    const bf16* vp = base + (size_t)(r0 + kk) * ld + (size_t)(nh + h) * hd;
    if (lane * 2 < hd) {
      const uint32_t va = *reinterpret_cast<const uint32_t*>(vp + lane * 2);
      o0 += p * bf16lo(va);
      o1 += p * bf16hi(va);
    }
  }
  if (lane * 2 < hd)
    *reinterpret_cast<uint32_t*>(out + ((size_t)b * n + t) * (size_t)(nh * hd) + (size_t)h * hd + lane * 2) = pack_bf16(o0, o1);
}

// ConvNeXt front: depthwise causal conv k=7 + LayerNorm(eps 1e-6) (…v2.py:230-232); one block per (b,t)
// (x_bs_rows / hist: the streaming decoder keeps 6 rows of history in front of every row's T new rows)
__global__ void dwconv_ln_kernel(const bf16* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                 const float* __restrict__ lnw, const float* __restrict__ lnb, bf16* __restrict__ y, int B, int T,
                                 int C, int x_bs_rows, int hist) {
  extern __shared__ float sh[];  // [C] conv outputs + 64 scratch
  const int bt = blockIdx.x;
  const int t = bt % T;
  const size_t xrow = (size_t)(bt / T) * x_bs_rows + hist + t;  // row of x that holds time step t of this batch row
  float s1 = 0.f, s2 = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = bias[c];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const int tt = t - 6 + j;
      if (tt >= -hist) acc += w[c * 7 + j] * bf2f(x[(xrow - 6 + j) * C + c]);
    }
    acc = rbf(acc);
    sh[c] = acc;
    s1 += acc;
    s2 += acc * acc;
  }
  float* red = sh + C;
  s1 = warp_sum(s1); s2 = warp_sum(s2);
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = s1; red[32 + (threadIdx.x >> 5)] = s2; }
  __syncthreads();
  float a = 0.f, q = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += red[i]; q += red[32 + i]; }
  const float mean = a / C;
  const float var = fmaxf(q / C - mean * mean, 0.f);
  const float inv = rsqrtf(var + 1e-6f);
  for (int c = threadIdx.x; c < C; c += blockDim.x) y[(size_t)bt * C + c] = f2bf((sh[c] - mean) * inv * lnw[c] + lnb[c]);
}

// after a packet: every history buffer keeps its last `hist` rows ([hist + T] rows were valid) at the front.
// One launch for all buffers; block = (entry, batch row); rows ascend so an overlapping move (T < hist) is safe.
struct RollEntry { bf16* p; int hist, T, C, bs_rows; };
struct RollTable { int n; RollEntry e[48]; };
__global__ void roll_history_kernel(RollTable tb, int B) {
  const RollEntry E = tb.e[blockIdx.x / B];
  const int b = blockIdx.x % B;
  bf16* base = E.p + (size_t)b * E.bs_rows * E.C;
  const int cv = E.C / 8;  // C % 16 == 0
  for (int r = 0; r < E.hist; ++r) {
    const uint4* src = reinterpret_cast<const uint4*>(base + (size_t)(E.T + r) * E.C);
    uint4* dst = reinterpret_cast<uint4*>(base + (size_t)r * E.C);
    for (int c = threadIdx.x; c < cv; c += blockDim.x) dst[c] = src[c];
    __syncthreads();  // row r complete before row r+1 may overwrite what a later source row aliases
  }
}

// final causal conv k=7, C -> 1, + clamp(-1,1) (…v2.py:863,884); one thread per output sample
__global__ void final_conv_kernel(const bf16* __restrict__ x, const float* __restrict__ w /*[7][C]*/, const float* __restrict__ bias_p,
                                  float* __restrict__ wav, int B, int T, int C, int x_bs_rows, int hist) {
  const size_t total = (size_t)B * T;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int t = (int)(i % T);
    const size_t xrow = (i / T) * (size_t)x_bs_rows + hist + t;
    float acc = __ldg(bias_p);
    for (int j = 0; j < 7; ++j) {
      const int tt = t - 6 + j;
      if (tt < -hist) continue;
      const bf16* xr = x + (xrow - 6 + j) * (size_t)C;
      for (int c = 0; c < C; c += 8) {
        const uint4 v = *reinterpret_cast<const uint4*>(xr + c);
        const float* wr = w + j * C + c;
        acc += bf16lo(v.x) * wr[0] + bf16hi(v.x) * wr[1] + bf16lo(v.y) * wr[2] + bf16hi(v.y) * wr[3] +
               bf16lo(v.z) * wr[4] + bf16hi(v.z) * wr[5] + bf16lo(v.w) * wr[6] + bf16hi(v.w) * wr[7];
      }
    }
    acc = rbf(acc);
    wav[i] = fminf(1.f, fmaxf(-1.f, acc));
  }
}

}  // namespace

// =================================================================================================
// cudaMalloc + zero fill queued on `stream` (work queued behind it there sees zeros); the allocation is recorded in
// `owned`, which its owner frees on destroy / close
template <class T>
static int dev_alloc(std::vector<void*>& owned, size_t bytes, cudaStream_t stream, T** out) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return q3_set_err("cudaMalloc(%zu B) failed: %s", bytes, cudaGetErrorString(e));
  owned.push_back(p);
  e = cudaMemsetAsync(p, 0, bytes, stream);
  if (e != cudaSuccess) return q3_set_err("cudaMemsetAsync(%zu B) failed: %s", bytes, cudaGetErrorString(e));
  *out = static_cast<T*>(p);
  return 0;
}

struct q3_codec {
  q3_codec_cfg cfg;
  std::map<std::string, DevTensor> t;
  std::vector<void*> allocs;
  bf16* buf[4] = {nullptr, nullptr, nullptr, nullptr};  // the one-shot forward's scratch (also in allocs)
  size_t buf_elems = 0;
  bool finalized = false;
  int total_up = 1;
  int launches = 0;
  struct Capture { int stage; bf16* dst; int64_t capacity; };
  std::vector<Capture> captures;  // test hook (q3_codec_debug_capture): stage ordinal -> destination of the next forward

  const DevTensor* get(const std::string& n) const {
    auto it = t.find(n);
    return it == t.end() ? nullptr : &it->second;
  }
};

extern "C" int q3_codec_create(const q3_codec_cfg* cfg, q3_codec** out) {
  Q3_REQUIRE(cfg && out, "null argument");
  Q3_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  Q3_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  Q3_REQUIRE(prop.major == 10, "this library is built for sm_100a (B200); device is sm_%d%d", prop.major, prop.minor);
  Q3_REQUIRE(cfg->head_dim % 2 == 0 && cfg->head_dim <= 64, "codec head_dim must be even and <= 64");
  Q3_REQUIRE(cfg->sliding_window <= 96, "sliding_window > 96 unsupported");
  Q3_REQUIRE(cfg->num_heads == cfg->num_kv_heads, "codec transformer is MHA in the reference config");
  Q3_REQUIRE(cfg->codebook_dim % 32 == 0 && cfg->latent_dim % 16 == 0 && cfg->hidden_size % 16 == 0 &&
                 cfg->intermediate_size % 16 == 0 && cfg->decoder_dim % 16 == 0,
             "channel counts must be multiples of 16");
  if (gemm_init()) return 1;
  q3_codec* c = new q3_codec();
  c->cfg = *cfg;
  c->total_up = 1;
  for (int i = 0; i < cfg->n_upsample_rates; ++i) c->total_up *= cfg->upsample_rates[i];
  for (int i = 0; i < cfg->n_upsampling_ratios; ++i) c->total_up *= cfg->upsampling_ratios[i];
  Q3_REQUIRE((cfg->decoder_dim >> cfg->n_upsample_rates) % 16 == 0, "final channel count must be a multiple of 16");
  *out = c;
  return 0;
}

extern "C" void q3_codec_destroy(q3_codec* c) {
  if (!c) return;
  for (void* p : c->allocs) cudaFree(p);
  delete c;
}

extern "C" int q3_codec_total_upsample(q3_codec* c) { return c ? c->total_up : 0; }
extern "C" int q3_codec_last_launch_count(q3_codec* c) { return c ? c->launches : 0; }

// Test hook (tests/ only): the next q3_codec_forward calls copy the bf16 [B][T_stage][C_stage] tensor of `stage` into
// dst_dev (at most `capacity` elements).  Stages: 0 pre_conv output, 1 pre-transformer output (after output_proj), 2 output
// of the upsample stack, 3 SnakeBeta(decoder.0 conv output) as fed to block 0, 4+i output of decoder block i.
// stage < 0 clears all captures.
extern "C" int q3_codec_debug_capture(q3_codec* c, int32_t stage, void* dst_dev, int64_t capacity) {
  Q3_REQUIRE(c, "null codec");
  if (stage < 0) { c->captures.clear(); return 0; }
  Q3_REQUIRE(dst_dev && capacity > 0, "bad capture destination");
  c->captures.push_back({stage, reinterpret_cast<bf16*>(dst_dev), capacity});
  return 0;
}

// Engine-native tensors (converted from the reference state_dict by the Python host, see INTEGRATION.md):
// shape[] / ndim describe the tensor; dtype is inferred from the name suffix: names ending in ".w" / "table" /
// "proj" / "norm" / "ln1" / "ln2" / "cos" / "sin" are bf16, everything else fp32.
static bool name_is_bf16(const std::string& n) {
  auto ends = [&](const char* s) { size_t l = strlen(s); return n.size() >= l && n.compare(n.size() - l, l, s) == 0; };
  if (ends(".dw.w") || ends("dec.out.w")) return false;
  return ends(".w") || ends(".table") || ends(".proj") || ends(".norm") || ends(".ln1") || ends(".ln2") || ends(".cos") ||
         ends(".sin");
}

extern "C" int q3_codec_load_tensor(q3_codec* c, const char* name, const void* dev, const int64_t* shape, int32_t ndim) {
  Q3_REQUIRE(c && name && dev && shape, "null argument");
  Q3_CUDA(cudaSetDevice(c->cfg.device));
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) n *= shape[i];
  DevTensor d;
  d.dtype = name_is_bf16(name) ? 0 : 1;
  d.numel = n;
  const size_t bytes = (size_t)n * (d.dtype == 0 ? 2 : 4);
  if (dev_alloc(c->allocs, (bytes + 255) & ~(size_t)255, nullptr /* ordered before the copy below */, &d.p)) return 1;
  Q3_CUDA(cudaMemcpy(d.p, dev, bytes, cudaMemcpyDeviceToDevice));
  c->t[name] = d;
  return 0;
}

#define NEED(var, nm, cnt)                                                                          \
  const DevTensor* var = c->get(nm);                                                                \
  Q3_REQUIRE(var, "codec: missing tensor %s", std::string(nm).c_str());                             \
  Q3_REQUIRE(var->numel == (int64_t)(cnt), "codec: tensor %s has %lld elements, expected %lld",     \
             std::string(nm).c_str(), (long long)var->numel, (long long)(cnt))

static int kpad(int k) { return (k + 63) / 64 * 64; }

extern "C" int q3_codec_finalize(q3_codec* c) {
  Q3_REQUIRE(c, "null codec");
  const q3_codec_cfg& g = c->cfg;
  // spot-check the tensors whose absence would otherwise only surface mid-forward
  {
    NEED(a, "rvq.table", (int64_t)g.num_quantizers * g.codebook_size * (g.codebook_dim / 2));
    NEED(b, "rvq.proj", (int64_t)g.codebook_dim * kpad(g.codebook_dim));
    NEED(d, "dec.out.w", (int64_t)7 * (g.decoder_dim >> g.n_upsample_rates));
    (void)a; (void)b; (void)d;
  }
  c->finalized = true;
  return 0;
}

// =================================================================================================
// Stateful streaming decoder (SURVEY §8f-2, §8b: q3_codec_stream_*).  Equal to the full causal forward over everything
// pushed so far (oracle/codec.py::StreamingDecoder is the spec; the reference's chunked_decode instead re-decodes 25
// frames of left context per chunk, …v2.py:886-896).  State per row: the last (k-1)*dilation input rows of every
// convolution with taps, the last input row of every k=2r ConvTranspose, and per transformer layer the rotated K and V
// of the last window-1 frames.  Every such tensor lives in a history-prefixed buffer [B][hist + T_cap][C]: its producer
// GEMM writes the new rows behind the history, its consumer GEMM reads through a TMA map whose taps reach back into the
// history (GemmViews), and one roll kernel per packet moves the last `hist` rows to the front.
// =================================================================================================
struct HistBuf {
  bf16* p = nullptr;
  int hist = 0, C = 0, cap = 0;                 // rows of history, channels, capacity in new rows
  int bs_rows() const { return hist + cap; }
  long long bs() const { return (long long)bs_rows() * C; }
  bf16* cur() const { return p + (size_t)hist * C; }  // first new row of batch row 0
};

struct q3_codec_stream {
  q3_codec* c = nullptr;
  int B = 0, nmax = 0, pos = 0;
  std::vector<void*> allocs;
  HistBuf pre, in, out;
  std::vector<HistBuf> dw, ct, kv;
  std::vector<std::vector<HistBuf>> c1;
  bf16* buf[4] = {nullptr, nullptr, nullptr, nullptr};
};

namespace {

struct Runner {
  q3_codec* c;
  cudaStream_t stream;
  int B;
  bool streaming;
  int err = 0;

  // one tap-GEMM: a [B][T][K] -> [B][T][N]; v: batch strides of outputs / residual that live in history buffers;
  // a_bs: batch stride of A in elements (0: T*K)
  void gemm(const bf16* a, int T, int K, const char* wname, int N, int ntaps, const int* shifts, GemmEpilogue ep,
            GemmViews v = {}, int64_t a_bs = 0) {
    if (err) return;
    const DevTensor* w = c->get(wname);
    const int Kp = kpad(K);
    if (!w || w->numel != (int64_t)N * ntaps * Kp) {
      err = q3_set_err("codec: tensor %s missing or wrong size (want %lld)", wname, (long long)N * ntaps * Kp);
      return;
    }
    if (ep.cmod == 0) ep.cmod = N;
    GemmPlan plan;
    const int mt = (T + 127) / 128;
    if (gemm_make_plan_v(&plan, a, B, T, K, K, a_bs ? a_bs : (int64_t)T * K, reinterpret_cast<const bf16*>(w->p), N, Kp, ntaps, shifts,
                         gemm_pick_bn(N, mt, B), ep, v)) { err = 1; return; }
    if (gemm_launch(plan, stream)) { err = 1; return; }
    c->launches++;
  }
  // the same with A read from a history buffer: the taps' negative shifts reach back into its history rows
  void gemm_h(const HistBuf& a, int T, const char* wname, int N, int ntaps, const int* shifts, GemmEpilogue ep,
              GemmViews v = {}) {
    v.a_rows = a.hist + T;
    v.a_row0 = a.hist;
    gemm(a.p, T, a.C, wname, N, ntaps, shifts, ep, v, a.bs());
  }
  // test hook: copy a stage's [B][T][C] bf16 tensor to every destination registered for `stage` (no launch, no sync).
  // One-shot only: in a stream the tensors have history rows between the batch rows.
  void capture(int stage, const bf16* x, int64_t elems) {
    if (err || streaming) return;
    for (const auto& cp : c->captures)
      if (cp.stage == stage) {
        const int64_t n = elems < cp.capacity ? elems : cp.capacity;
        if (cudaMemcpyAsync(cp.dst, x, (size_t)n * 2, cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
          err = q3_set_err("codec: capture of stage %d failed", stage);
      }
  }
  const float* f32(const std::string& n, int64_t cnt) {
    const DevTensor* d = c->get(n);
    if (!d || d->numel != cnt || d->dtype != 1) { if (!err) err = q3_set_err("codec: fp32 tensor %s missing/wrong size", n.c_str()); return nullptr; }
    return reinterpret_cast<const float*>(d->p);
  }
  const bf16* b16(const std::string& n, int64_t cnt) {
    const DevTensor* d = c->get(n);
    if (!d || d->numel != cnt || d->dtype != 0) { if (!err) err = q3_set_err("codec: bf16 tensor %s missing/wrong size", n.c_str()); return nullptr; }
    return reinterpret_cast<const bf16*>(d->p);
  }
};

// per-(b, frame) element high-water mark of a scratch buffer over all stages
size_t scratch_per_frame(const q3_codec_cfg& g) {
  size_t per_frame = std::max<size_t>({(size_t)3 * g.num_heads * g.head_dim, (size_t)2 * g.intermediate_size,
                                       (size_t)g.latent_dim, (size_t)g.codebook_dim});
  size_t up = 1;
  for (int i = 0; i < g.n_upsampling_ratios; ++i) { up *= g.upsampling_ratios[i]; per_frame = std::max(per_frame, up * 4 * g.latent_dim); }
  per_frame = std::max(per_frame, up * (size_t)g.decoder_dim);
  int ch = g.decoder_dim;
  for (int i = 0; i < g.n_upsample_rates; ++i) { up *= g.upsample_rates[i]; ch /= 2; per_frame = std::max(per_frame, up * (size_t)ch); }
  return per_frame;
}

// The decoder: codes [B][K][T] -> wav [B][T * total_upsample], through the four scratch buffers `buf`.  s == nullptr is
// the one-shot forward; otherwise these are the next T frames of stream s.  The one-shot forward is the stream with
// zero history: every tensor a stream keeps history for goes through place(), which returns the stream's own buffer,
// or in one-shot mode the scratch slot the choreography below assigns, as a view without history (every GemmViews field
// then resolves to its contiguous default).  Stream mode only ever replaces scratch slots by private buffers, so it only removes
// aliasing pairs: a slot assignment that is hazard-free for the one-shot forward is hazard-free for the stream.
int decode(q3_codec* c, q3_codec_stream* s, bf16* const buf[4], const int32_t* codes, int B, int T, float* wav,
           cudaStream_t stream) {
  const q3_codec_cfg& g = c->cfg;
  const int Cl = g.latent_dim, Hh = g.hidden_size, nh = g.num_heads, hd = g.head_dim, I = g.intermediate_size;
  bf16 *X = buf[0], *Y = buf[1], *Z = buf[2], *W = buf[3];
  Runner R{c, stream, B, s != nullptr};
  c->launches = 0;
  const int zero = 0;
  GemmEpilogue none{};
  auto place = [](const HistBuf* own, bf16* slot, int rows, int C) { return own ? *own : HistBuf{slot, 0, C, rows}; };
  RollTable roll{};
  auto add_roll = [&](const HistBuf& h, int rows) {
    if (h.hist > 0) roll.e[roll.n++] = RollEntry{h.p, h.hist, rows, h.C, h.bs_rows()};
  };

  // ---- RVQ decode -> X [B][T][codebook_dim]; projection; pre_conv k=3 (…v2.py:839-843,874)
  const int D = g.codebook_dim / 2;
  rvq_gather_kernel<<<B * T, 128, 0, stream>>>(codes, R.b16("rvq.table", (int64_t)g.num_quantizers * g.codebook_size * D), X, B,
                                               g.num_quantizers, T, D, g.codebook_size);
  c->launches++;
  if (R.err) return 1;
  const HistBuf pre = place(s ? &s->pre : nullptr, Y, T, g.codebook_dim);
  { GemmEpilogue e = none; e.out_raw = pre.cur(); GemmViews v; v.raw_bs = pre.bs();
    R.gemm(X, T, g.codebook_dim, "rvq.proj", g.codebook_dim, 1, &zero, e, v); }
  { const int sh[3] = {-2, -1, 0}; GemmEpilogue e = none; e.bias = R.f32("pre_conv.b", Cl); e.out_raw = X;
    R.gemm_h(pre, T, "pre_conv.w", Cl, 3, sh, e); }
  add_roll(pre, T);
  R.capture(0, X, (int64_t)B * T * Cl);
  // ---- pre_transformer (…v2.py:501-575)
  { GemmEpilogue e = none; e.bias = R.f32("tr.in.b", Hh); e.out_raw = Y; R.gemm(X, T, Cl, "tr.in.w", Hh, 1, &zero, e); }
  bf16* xres = Y;  // residual stream [B][T][Hh]
  const int rows = B * T;
  const int pos0 = s ? s->pos : 0;
  for (int l = 0; l < g.num_layers && !R.err; ++l) {
    const std::string p = "tr." + std::to_string(l);
    rmsnorm_rows_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(xres, R.b16(p + ".ln1", Hh), X, rows, Hh, g.rms_eps);
    { GemmEpilogue e = none; e.out_raw = Z; R.gemm(X, T, Hh, (p + ".qkv.w").c_str(), 3 * nh * hd, 1, &zero, e); }
    // K/V rows: the stream's window buffer of this layer, which RoPE appends the new rows to; in one-shot mode the k and
    // v heads of qkv itself, read in place (C = 3*nh*hd is then the row pitch)
    const HistBuf* win = s ? &s->kv[l] : nullptr;
    const HistBuf kv = win ? *win : HistBuf{Z + nh * hd, 0, 3 * nh * hd, T};
    rope_kernel<<<win ? 148 : 296, 256, 0, stream>>>(Z, R.b16("rope.cos", (int64_t)g.max_frames * (hd / 2)),
                                                     R.b16("rope.sin", (int64_t)g.max_frames * (hd / 2)), win ? win->p : nullptr,
                                                     kv.hist, kv.bs_rows(), B, T, nh, hd, pos0);
    window_attention_kernel<<<(rows * nh + 7) / 8, 256, 0, stream>>>(Z, kv.p, kv.C, kv.bs_rows(), kv.hist, pos0, X, B, T, nh,
                                                                     hd, g.sliding_window);
    add_roll(kv, T);
    { GemmEpilogue e = none; e.scale = R.f32(p + ".ls1", Hh); e.resid = xres; e.out_raw = W;
      R.gemm(X, T, nh * hd, (p + ".o.w").c_str(), Hh, 1, &zero, e); }
    rmsnorm_rows_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(W, R.b16(p + ".ln2", Hh), X, rows, Hh, g.rms_eps);
    { GemmEpilogue e = none; e.act = ACT_SWIGLU_PAIR; e.out_act = Z; R.gemm(X, T, Hh, (p + ".gate_up.w").c_str(), 2 * I, 1, &zero, e); }
    { GemmEpilogue e = none; e.scale = R.f32(p + ".ls2", Hh); e.resid = W; e.out_raw = xres;
      R.gemm(Z, T, I, (p + ".down.w").c_str(), Hh, 1, &zero, e); }
    c->launches += 4;
  }
  rmsnorm_rows_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(xres, R.b16("tr.norm", Hh), X, rows, Hh, g.rms_eps);
  c->launches++;
  { GemmEpilogue e = none; e.bias = R.f32("tr.out.b", Cl); e.out_raw = Z; R.gemm(X, T, Hh, "tr.out.w", Cl, 1, &zero, e); }
  R.capture(1, Z, (int64_t)B * T * Cl);
  // ---- upsample: ConvT(k=s=f) + ConvNeXt (…v2.py:845-855,878-880); each stage reads its input from Z and writes its
  // output back there; the last stage's output is decoder.0's input
  HistBuf up{Z, 0, Cl, T};  // [B][Tc][Cl]
  int Tc = T;
  for (int i = 0; i < g.n_upsampling_ratios && !R.err; ++i) {
    const int f = g.upsampling_ratios[i];
    const std::string p = "up." + std::to_string(i);
    const HistBuf u = place(s ? &s->dw[i] : nullptr, Y, Tc * f, Cl);
    { GemmEpilogue e = none; e.bias = R.f32(p + ".ct.b", Cl); e.cmod = Cl; e.out_raw = u.cur(); GemmViews v; v.raw_bs = u.bs();
      R.gemm(Z, Tc, Cl, (p + ".ct.w").c_str(), f * Cl, 1, &zero, e, v); }
    Tc *= f;
    const float *dww = R.f32(p + ".dw.w", (int64_t)Cl * 7), *dwb = R.f32(p + ".dw.b", Cl), *lw = R.f32(p + ".ln_g", Cl),
                *lb = R.f32(p + ".ln_beta", Cl);
    if (R.err) break;
    dwconv_ln_kernel<<<B * Tc, 256, (Cl + 64) * sizeof(float), stream>>>(u.p, dww, dwb, lw, lb, X, B, Tc, Cl, u.bs_rows(), u.hist);
    c->launches++;
    { GemmEpilogue e = none; e.bias = R.f32(p + ".pw1.b", 4 * Cl); e.act = ACT_GELU; e.out_act = W;
      R.gemm(X, Tc, Cl, (p + ".pw1.w").c_str(), 4 * Cl, 1, &zero, e); }
    up = place(s && i + 1 == g.n_upsampling_ratios ? &s->in : nullptr, Z, Tc, Cl);
    { GemmEpilogue e = none; e.bias = R.f32(p + ".pw2.b", Cl); e.scale = R.f32(p + ".gamma", Cl); e.resid = u.cur(); e.out_raw = up.cur();
      GemmViews v; v.resid_bs = u.bs(); v.raw_bs = up.bs();
      R.gemm(W, Tc, 4 * Cl, (p + ".pw2.w").c_str(), Cl, 1, &zero, e, v); }
    add_roll(u, Tc);
  }
  R.capture(2, up.p, (int64_t)B * Tc * Cl);
  // ---- decoder.0: conv k7 latent -> decoder_dim; epilogue applies block 0's SnakeBeta (…v2.py:857,646)
  const int nb = g.n_upsample_rates;
  // the SnakeBeta-activated input of block bi's ConvTranspose; bi == nb: of the final conv
  auto block_in = [&](int bi, bf16* slot, int rows_, int C_) {
    return place(!s ? nullptr : bi < nb ? &s->ct[bi] : &s->out, slot, rows_, C_);
  };
  int C = g.decoder_dim;
  bf16* act = X;  // snake-activated input of the next conv
  HistBuf a = block_in(0, act, Tc, C);
  {
    const int sh[7] = {-6, -5, -4, -3, -2, -1, 0};
    GemmEpilogue e = none; e.bias = R.f32("dec.in.b", C); e.act = ACT_SNAKE; e.snake_ea = R.f32("dec.0.snake_ea", C);
    e.snake_ib = R.f32("dec.0.snake_ib", C); e.out_act = a.cur();
    GemmViews v; v.act_bs = a.bs();
    R.gemm_h(up, Tc, "dec.in.w", C, 7, sh, e, v);
  }
  add_roll(up, Tc);
  R.capture(3, a.p, (int64_t)B * Tc * C);  // SnakeBeta(decoder.0 output) with block 0's leading activation
  // ---- decoder blocks (…v2.py:638-658, :619-635)
  bf16 *y = Y, *tmp = Z, *act2 = W;
  for (int bi = 0; bi < nb && !R.err; ++bi) {
    const int r = g.upsample_rates[bi];
    const int Co = C / 2;
    const std::string p = "dec." + std::to_string(bi);
    const HistBuf a1 = place(s ? &s->c1[bi][0] : nullptr, act2, Tc * r, Co);
    {
      const int sh[2] = {0, -1};
      GemmEpilogue e = none; e.bias = R.f32(p + ".ct.b", Co); e.cmod = Co; e.out_raw = y; e.act = ACT_SNAKE;
      e.snake_ea = R.f32(p + ".0.s1_ea", Co); e.snake_ib = R.f32(p + ".0.s1_ib", Co); e.out_act = a1.cur();
      GemmViews v; v.act_bs = a1.bs();
      R.gemm_h(a, Tc, (p + ".ct.w").c_str(), r * Co, 2, sh, e, v);
    }
    add_roll(a, Tc);
    Tc *= r;
    C = Co;
    std::swap(act, act2);  // act now holds snake1(y)
    a = a1;
    for (int u = 0; u < 3 && !R.err; ++u) {
      const int dil = u == 0 ? 1 : (u == 1 ? 3 : 9);
      const std::string q = p + "." + std::to_string(u);
      {
        int sh[7];
        for (int j = 0; j < 7; ++j) sh[j] = -(6 - j) * dil;
        GemmEpilogue e = none; e.bias = R.f32(q + ".c1.b", C); e.act = ACT_SNAKE; e.snake_ea = R.f32(q + ".s2_ea", C);
        e.snake_ib = R.f32(q + ".s2_ib", C); e.out_act = tmp;
        R.gemm_h(a, Tc, (q + ".c1.w").c_str(), C, 7, sh, e);
      }
      add_roll(a, Tc);
      {
        // next activation: next unit's act1, or the next block's leading snake, or the final snake
        std::string nx = (u < 2) ? (p + "." + std::to_string(u + 1) + ".s1")
                                 : (bi + 1 < nb ? ("dec." + std::to_string(bi + 1) + ".snake") : std::string("dec.out.snake"));
        a = (u < 2) ? place(s ? &s->c1[bi][u + 1] : nullptr, act, Tc, C) : block_in(bi + 1, act, Tc, C);
        GemmEpilogue e = none; e.bias = R.f32(q + ".c2.b", C); e.resid = y; e.out_raw = act2 /*new y*/; e.act = ACT_SNAKE;
        e.snake_ea = R.f32(nx + "_ea", C); e.snake_ib = R.f32(nx + "_ib", C); e.out_act = a.cur();
        GemmViews v; v.act_bs = a.bs();
        // out_act overwrites `act` (this GEMM's input is tmp, its residual is y) — safe
        R.gemm(tmp, Tc, C, (q + ".c2.w").c_str(), C, 1, &zero, e, v);
        std::swap(y, act2);  // y <- new residual stream
      }
    }
    R.capture(4 + bi, y, (int64_t)B * Tc * C);  // the block's output (residual stream after its three units)
  }
  if (R.err) return 1;
  // ---- final conv + clamp
  {
    const float* w = R.f32("dec.out.w", (int64_t)7 * C);
    const float* bsrc = R.f32("dec.out.b", 1);
    if (R.err) return 1;
    final_conv_kernel<<<1184, 256, 0, stream>>>(a.p, w, bsrc, wav, B, Tc, C, a.bs_rows(), a.hist);  // bias read on the device: no host round trip
    c->launches++;
  }
  add_roll(a, Tc);
  if (roll.n) {  // stream mode: keep the last `hist` rows of every history buffer for the next packet
    Q3_REQUIRE(roll.n <= 48, "roll table overflow");
    roll_history_kernel<<<roll.n * B, 128, 0, stream>>>(roll, B);
    c->launches++;
  }
  Q3_CUDA(cudaGetLastError());
  return R.err;
}

}  // namespace

extern "C" int q3_codec_forward(q3_codec* c, const int32_t* codes_dev, int32_t B, int32_t T, float* wav_dev, void* stream_) {
  Q3_REQUIRE(c && c->finalized, "codec not finalized");
  Q3_REQUIRE(codes_dev && wav_dev && B >= 1 && T >= 1, "bad arguments");
  Q3_REQUIRE(T <= c->cfg.max_frames, "T=%d exceeds max_frames=%d", T, c->cfg.max_frames);
  Q3_CUDA(cudaSetDevice(c->cfg.device));
  cudaStream_t stream = (cudaStream_t)stream_;
  const size_t need = scratch_per_frame(c->cfg) * (size_t)B * T;
  if (need > c->buf_elems) {
    // replace the scratch; cudaFree waits for work still using the old buffers
    for (bf16*& p : c->buf) {
      if (!p) continue;
      c->allocs.erase(std::find(c->allocs.begin(), c->allocs.end(), (void*)p));
      Q3_CUDA(cudaFree(p));
      p = nullptr;
    }
    c->buf_elems = 0;
    for (bf16*& p : c->buf)
      if (dev_alloc(c->allocs, need * 2 + 1024, stream, &p)) return 1;
    c->buf_elems = need;
  }
  return decode(c, nullptr, c->buf, codes_dev, B, T, wav_dev, stream);
}

extern "C" int q3_codec_stream_open(q3_codec* c, int32_t B, int32_t max_packet_frames, q3_codec_stream** out) {
  Q3_REQUIRE(c && c->finalized && out, "codec not finalized");
  Q3_REQUIRE(B >= 1 && B <= c->cfg.max_batch && max_packet_frames >= 1 && max_packet_frames <= c->cfg.max_frames, "bad arguments");
  const q3_codec_cfg& g = c->cfg;
  // decoder.0 reads its history from the last upsampling stage's output buffer
  Q3_REQUIRE(g.n_upsampling_ratios >= 1, "streaming decoder expects at least one upsampling stage");
  Q3_CUDA(cudaSetDevice(g.device));
  q3_codec_stream* s = new q3_codec_stream();
  s->c = c; s->B = B; s->nmax = max_packet_frames;
  const int n = max_packet_frames, Cl = g.latent_dim, nh = g.num_heads, hd = g.head_dim;
  // zero history == the causal left padding of a fresh stream
  auto hist_alloc = [&](HistBuf* h, int hist, int C, int cap) {
    h->hist = hist; h->C = C; h->cap = cap;
    return dev_alloc(s->allocs, (size_t)B * h->bs_rows() * C * 2 + 256, nullptr, &h->p);
  };
  int rc = hist_alloc(&s->pre, 2, g.codebook_dim, n);
  s->kv.resize(g.num_layers);
  for (int l = 0; l < g.num_layers && !rc; ++l) rc = hist_alloc(&s->kv[l], g.sliding_window - 1, 2 * nh * hd, n);
  int Tc = n;
  s->dw.resize(g.n_upsampling_ratios);
  for (int i = 0; i < g.n_upsampling_ratios && !rc; ++i) { Tc *= g.upsampling_ratios[i]; rc = hist_alloc(&s->dw[i], 6, Cl, Tc); }
  if (!rc) rc = hist_alloc(&s->in, 6, Cl, Tc);
  int C = g.decoder_dim;
  s->ct.resize(g.n_upsample_rates);
  s->c1.resize(g.n_upsample_rates);
  for (int bi = 0; bi < g.n_upsample_rates && !rc; ++bi) {
    rc = hist_alloc(&s->ct[bi], 1, C, Tc);
    Tc *= g.upsample_rates[bi];
    C /= 2;
    s->c1[bi].resize(3);
    const int dil[3] = {1, 3, 9};
    for (int u = 0; u < 3 && !rc; ++u) rc = hist_alloc(&s->c1[bi][u], 6 * dil[u], C, Tc);
  }
  if (!rc) rc = hist_alloc(&s->out, 6, C, Tc);
  for (int i = 0; i < 4 && !rc; ++i) rc = dev_alloc(s->allocs, scratch_per_frame(g) * (size_t)B * n * 2 + 1024, nullptr, &s->buf[i]);
  if (rc) { for (void* p : s->allocs) cudaFree(p); delete s; return 1; }
  Q3_CUDA(cudaDeviceSynchronize());
  *out = s;
  return 0;
}

extern "C" void q3_codec_stream_close(q3_codec_stream* s) {
  if (!s) return;
  for (void* p : s->allocs) cudaFree(p);
  delete s;
}

extern "C" int q3_codec_stream_position(q3_codec_stream* s) { return s ? s->pos : -1; }

// next n frames of every row: codes_dev int32 [B][K][n] -> wav_dev fp32 [B][n * total_upsample]
extern "C" int q3_codec_stream_step(q3_codec_stream* s, const int32_t* codes_dev, int32_t n, float* wav_dev, void* stream_) {
  Q3_REQUIRE(s && codes_dev && wav_dev, "null argument");
  Q3_REQUIRE(n >= 1 && n <= s->nmax, "packet of %d frames (max %d)", n, s->nmax);
  const q3_codec_cfg& g = s->c->cfg;
  Q3_REQUIRE(s->pos + n <= g.max_frames, "stream position %d + %d exceeds the RoPE table (max_frames %d)", s->pos, n, g.max_frames);
  Q3_CUDA(cudaSetDevice(g.device));
  if (decode(s->c, s, s->buf, codes_dev, s->B, n, wav_dev, (cudaStream_t)stream_)) return 1;
  s->pos += n;
  return 0;
}

// forget everything: the next packet starts a new utterance
extern "C" int q3_codec_stream_reset(q3_codec_stream* s, void* stream_) {
  Q3_REQUIRE(s, "null stream");
  cudaStream_t stream = (cudaStream_t)stream_;
  auto z = [&](const HistBuf& h) { return cudaMemsetAsync(h.p, 0, (size_t)s->B * h.bs_rows() * h.C * 2, stream); };
  Q3_CUDA(z(s->pre)); Q3_CUDA(z(s->in)); Q3_CUDA(z(s->out));
  for (auto& h : s->dw) Q3_CUDA(z(h));
  for (auto& h : s->ct) Q3_CUDA(z(h));
  for (auto& h : s->kv) Q3_CUDA(z(h));
  for (auto& v : s->c1) for (auto& h : v) Q3_CUDA(z(h));
  s->pos = 0;
  return 0;
}
