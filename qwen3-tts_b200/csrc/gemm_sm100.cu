// tcgen05 tap-GEMM kernel (see gemm_sm100.cuh).  Warp-specialised and PERSISTENT: a CTA walks 128 x bn output tiles
// (tile = blockIdx.x, += gridDim.x) with TWO accumulators in TMEM, so the epilogue of tile i (tcgen05.ld, bias /
// LayerScale / residual / SnakeBeta / GELU / SwiGLU, bf16 stores) overlaps the TMA + MMA mainloop of tile i+1:
//   warp 0  : TMA producer (A tile via a 3-D map with a per-tap row shift, W tile via a 2-D map), 4-stage ring that
//             keeps running across tiles
//   warp 1  : TMEM allocator + single-thread tcgen05.mma issuer (M=128, N=bn, K=16, bf16 -> fp32 in TMEM); waits for
//             the accumulator it is about to overwrite (tmem_empty), commits tmem_full when a tile is complete
//   warps 2-17: epilogue — one output row per thread, four warps per TMEM lane quadrant (interleaved 16-column chunks);
//             arrive on tmem_empty when the accumulator has been read.
#include "gemm_sm100.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace {

constexpr int BM = 128;
constexpr int BK = 64;           // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int MAX_STAGES = 4;
constexpr int A_BYTES = BM * BK * 2;        // 16 KB
constexpr int SMEM_OPTIN = 232448;          // 227 KB
// epilogue staging, per TMEM lane quadrant: X0, X1 (residual in / pre-activation out, alternating per step) and Y
// (activated out), each 32 rows x 128 B (64 bf16 columns) with the 16-byte chunks XOR-swizzled by the row
constexpr int EPI_BUF = 32 * 128;
constexpr int EPI_Q_BYTES = 3 * EPI_BUF;
constexpr int EPI_BYTES = 4 * EPI_Q_BYTES;  // 48 KB
constexpr int BAR_BYTES = 256;              // full[S], empty[S], tmem_full[2], tmem_empty[2], tmem slot
constexpr int EPI_WARPS = 16;                        // four per TMEM lane quadrant: the epilogue (tcgen05.ld + SnakeBeta / GELU /
                                                     // residual + stores) is what bounds the short-K convolutions (measured: 4 warps
                                                     // 28.5 ms, 8 warps 18.3 ms for the 8 x 125-frame codec)
constexpr int GEMM_THREADS = 64 + 32 * EPI_WARPS;    // producer warp, MMA warp, epilogue warps
__host__ __device__ inline int stage_bytes_for(int bn) { return A_BYTES + ((bn * BK * 2 + 1023) & ~1023); }
inline int stages_for(int bn) { return std::min(MAX_STAGES, (SMEM_OPTIN - 1024 - BAR_BYTES - EPI_BYTES) / stage_bytes_for(bn)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = clock64();
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    if (clock64() - t0 > 4000000000LL) __trap();  // never hang the box on a protocol bug
  }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"): 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);        // start address
  d |= (uint64_t)1 << 16;                          // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset
  d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }

// sin for the SnakeBeta epilogue: Cody-Waite reduction to [-pi, pi] (k * 6.28125 is exact for |k| < 2^15), then the SFU
// (MUFU.SIN, abs error 2^-21.4 on that interval).  The result is squared, scaled and rounded to bf16 (2^-9 relative), so
// this is far inside the output's resolution for every argument below ~1e4; sinf()'s 20-instruction polynomial made
// the epilogue of the short-K decoder convolutions as long as their mainloop.
__device__ __forceinline__ float snake_sin(float a) {
  const float k = (fmaf(a, 0.15915494309189535f, 12582912.f)) - 12582912.f;  // rint for |a/2pi| < 2^22, on the FMA pipe (FRND is quarter-rate)
  float r = fmaf(-k, 6.28125f, a);
  r = fmaf(-k, 1.9353071795864769e-3f, r);
  return __sinf(r);
}

__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// 16 consecutive per-channel fp32 parameters (the channel index is a multiple of 16 and the vectors are 16-byte aligned)
__device__ __forceinline__ void ldg16(const float* ptr, float (&o)[16]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(ptr) + i);
    o[4 * i] = t.x; o[4 * i + 1] = t.y; o[4 * i + 2] = t.z; o[4 * i + 3] = t.w;
  }
}

// Round 16 values to bf16 and back (a PyTorch bf16 intermediate), two at a time through the packing convert
// (F2FP.PACK_AB) — the scalar F2F.BF16.F32 goes through the quarter-rate XU pipe.  xp keeps the packed pairs.
__device__ __forceinline__ void round16(float (&x)[16], uint32_t (&xp)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    xp[i] = pack_bf16(x[2 * i], x[2 * i + 1]);
    x[2 * i] = bf16lo(xp[i]);
    x[2 * i + 1] = bf16hi(xp[i]);
  }
}

// ACT is a template parameter on purpose: with a run-time activation code ptxas if-converts the three activation
// branches and evaluates erff() AND sin() for every element (measured: 55 instructions per output element).
template <int ACT>
__global__ void __launch_bounds__(GEMM_THREADS, 1) tap_gemm_kernel(const __grid_constant__ GemmPlan p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int STAGES = p.nst, STAGE_BYTES = stage_bytes_for(p.bn);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);  // full[S], empty[S], tmem_full[2], tmem_empty[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 4);
  unsigned char* epi_smem = smem + STAGES * STAGE_BYTES + BAR_BYTES;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kpb = p.Kp / BK;
  const int nkb = p.ntaps * kpb;
  const int mtiles = (p.T + BM - 1) / BM, ntiles = (p.N + p.bn - 1) / p.bn;
  const int total = mtiles * ntiles * p.B;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + MAX_STAGES), tfull0 = smem_u32(bars + 2 * MAX_STAGES),
                 tempty0 = smem_u32(bars + 2 * MAX_STAGES + 2);
  const uint32_t b_bytes = (uint32_t)p.bn * BK * 2;
  uint32_t acc_cols = 32;  // columns of one accumulator (power of two >= bn); two accumulators are allocated
  while (acc_cols < (uint32_t)p.bn) acc_cols <<= 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmW) : "memory");
    for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull0 + 8 * a, 1); mbar_init(tempty0 + 8 * a, EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(2 * acc_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0, round = 0;  // ring slot and how many times the ring has wrapped, over all tiles
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int nt = tile % ntiles, mt = (tile / ntiles) % mtiles, b = tile / (ntiles * mtiles);
        const int m0 = mt * BM, n0 = nt * p.bn;
        for (int kb = 0; kb < nkb; ++kb) {
          if (round > 0) mbar_wait(empty0 + 8 * s, (round - 1) & 1);
          const int tap = kb / kpb, k0 = (kb - tap * kpb) * BK;
          const uint32_t sa = smem_u32(smem + s * STAGE_BYTES), sb = sa + A_BYTES;
          mbar_expect_tx(full0 + 8 * s, A_BYTES + b_bytes);
          tma_load_3d(sa, &p.tmA, k0, m0 + p.shift[tap] + p.a_row0, b, full0 + 8 * s);
          tma_load_2d(sb, &p.tmW, tap * p.Kp + k0, n0, full0 + 8 * s);
          if (++s == STAGES) { s = 0; ++round; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // instruction descriptor: D=f32, A=B=bf16, both K-major, N=bn, M=128
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int s = 0, round = 0, lt = 0;  // ring position; local tile counter (accumulator = lt & 1)
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++lt) {
        const int acc = lt & 1;
        if (lt >= 2) {  // the epilogue must have drained this accumulator (tile lt-2)
          mbar_wait(tempty0 + 8 * acc, ((lt >> 1) - 1) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const uint32_t tacc = tmem_base + (uint32_t)acc * acc_cols;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(full0 + 8 * s, round & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa = smem_u32(smem + s * STAGE_BYTES), sb = sa + A_BYTES;
          const uint64_t ad = make_sdesc(sa), bd = make_sdesc(sb);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 bf16 = 32 B inside the 128 B swizzle row: +2 in the (>>4) start-address field
            umma_bf16(tacc, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc, (kb | k) != 0);
          }
          umma_commit(empty0 + 8 * s);                     // frees the smem slot once these MMAs have read it
          if (kb == nkb - 1) umma_commit(tfull0 + 8 * acc);  // accumulator complete
          if (++s == STAGES) { s = 0; ++round; }
        }
      }
    }
  } else {
    // ---- epilogue.  Warp w owns TMEM lanes [32*(w%4), +32) (a hardware rule), one output row per thread; the four
    // warps of a lane quadrant take the four 16-column chunks of one 64-column group per step.  Row-per-thread global
    // accesses touch 32 different 128-byte lines per instruction, which made the LSU — not DRAM — the bound of the k=1
    // convolutions (7-tap and 1-tap convolutions with the same output took the same time).  So the quadrant's 32 x 64
    // bf16 block goes through a swizzled shared-memory buffer: residual rows arrive by coalesced cp.async one step
    // ahead, results leave as 128-byte row segments (4 lines per store instruction instead of 32).
    const int q = warp & 3;
    const int j = (warp - 2) >> 2;           // 16-column chunk of the group
    const int tq = j * 32 + lane;            // thread index inside the quadrant group (128 threads, named barrier 1+q)
    const GemmEpilogue& E = p.ep;
    constexpr bool swiglu = ACT == ACT_SWIGLU_PAIR || ACT == ACT_SWIGLU_BLK8;
    const uint32_t X0 = smem_u32(epi_smem + q * EPI_Q_BYTES);  // X[k] = X0 + k * EPI_BUF (shared-space addresses)
    const uint32_t Y = X0 + 2 * EPI_BUF;
    const int ngroups = (p.bn + 63) >> 6;
    // the two 16-byte items of the quadrant block this thread moves in the cooperative (coalesced) copies
    const int it_row0 = tq >> 3, it_chunk = tq & 7;  // second item: row + 16
    // own slots (row = lane): chunks 2j and 2j+1
    const uint32_t own0 = (uint32_t)lane * 128u + (uint32_t)(((2 * j) ^ (lane & 7)) << 4),
                   own1 = (uint32_t)lane * 128u + (uint32_t)(((2 * j + 1) ^ (lane & 7)) << 4);
    auto qbar = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory"); };
    auto tile_coords = [&](int t, int& b_, int& m0_, int& n0_) {
      const int nt_ = t % ntiles, mt_ = (t / ntiles) % mtiles;
      b_ = t / (ntiles * mtiles); m0_ = mt_ * BM; n0_ = nt_ * p.bn;
    };
    // coalesced residual fetch of group g of the tile at (b_, m0_, n0_) into buffer `dst`; always commits a group
    auto issue_resid = [&](bool valid, int b_, int m0_, int n0_, int g, uint32_t dst) {
      const int col = g * 64 + it_chunk * 8;
      if (valid && col < p.bn && n0_ + col < p.N) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int r = it_row0 + 16 * i, m_ = m0_ + q * 32 + r;
          if (m_ < p.T) {
            const bf16* src = E.resid + (size_t)b_ * (size_t)p.resid_bs + (size_t)m_ * (size_t)p.N + n0_ + col;
            const uint32_t d = dst + r * 128 + ((it_chunk ^ (r & 7)) << 4);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto store_rows = [&](uint32_t src, bf16* out, long long bs, int b_, int m0_, int n0_, int g) {
      const int col = g * 64 + it_chunk * 8;
      if (col >= p.bn || n0_ + col >= p.N) return;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int r = it_row0 + 16 * i, m_ = m0_ + q * 32 + r;
        if (m_ < p.T) {
          const uint4 v = lds128(src + r * 128 + ((it_chunk ^ (r & 7)) << 4));
          *reinterpret_cast<uint4*>(out + (size_t)b_ * (size_t)bs + (size_t)m_ * (size_t)p.N + n0_ + col) = v;
        }
      }
    };
    int lt = 0, step = 0;
    int b = 0, m0 = 0, n0 = 0, nb = 0, nm0 = 0, nn0 = 0;  // this tile's and the next tile's coordinates (the divisions happen once per tile)
    if ((int)blockIdx.x < total) tile_coords(blockIdx.x, nb, nm0, nn0);
    if (!swiglu && E.resid) issue_resid((int)blockIdx.x < total, nb, nm0, nn0, 0, X0);
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++lt) {
    const int acc = lt & 1;
    b = nb; m0 = nm0; n0 = nn0;
    const bool more = tile + (int)gridDim.x < total;
    if (more) tile_coords(tile + gridDim.x, nb, nm0, nn0);
    const int m = m0 + q * 32 + lane;
    const bool row_ok = m < p.T;
    mbar_wait(tfull0 + 8 * acc, (lt >> 1) & 1);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tacc = tmem_base + (uint32_t)acc * acc_cols + ((uint32_t)(q * 32) << 16);
    if constexpr (swiglu) {
      // gated-MLP epilogues (transformer layers only, T = frames): halves the width, written directly
      for (int c0 = j * 16; c0 < p.bn; c0 += 64) {
        uint32_t v[16];
        tmem_ld16(tacc + (uint32_t)c0, v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const int n = n0 + c0;
        if (!row_ok || n >= p.N) continue;
        float x[16];
        const int ch = n % E.cmod;
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = rbf(__uint_as_float(v[i]) + (E.bias ? E.bias[ch + i] : 0.f));
        float y[8];
        if constexpr (ACT == ACT_SWIGLU_BLK8) {  // 16 columns = gate[8j..8j+7] | up[8j..8j+7] (the AR engine's gate_up row interleave)
#pragma unroll
          for (int i = 0; i < 8; ++i) { const float gt = x[i], u = x[8 + i]; y[i] = rbf(gt / (1.f + __expf(-gt))) * u; }
        } else {                         // columns (2i, 2i+1) = (gate_i, up_i)
#pragma unroll
          for (int i = 0; i < 8; ++i) { const float gt = x[2 * i], u = x[2 * i + 1]; y[i] = rbf(gt / (1.f + __expf(-gt))) * u; }
        }
        uint4 o;
        o.x = pack_bf16(y[0], y[1]); o.y = pack_bf16(y[2], y[3]); o.z = pack_bf16(y[4], y[5]); o.w = pack_bf16(y[6], y[7]);
        *reinterpret_cast<uint4*>(E.out_act + (size_t)b * (size_t)p.act_bs + (size_t)m * (size_t)(p.N / 2) + n / 2) = o;
      }
    } else {
      uint32_t v[16];
      for (int g = 0; g < ngroups; ++g, ++step) {
        const uint32_t Xc = X0 + (step & 1) * EPI_BUF;
        const int c0 = g * 64 + j * 16, n = n0 + c0;
        const bool have = c0 < p.bn && n < p.N;
        if (g == 0 && have) tmem_ld16(tacc + (uint32_t)c0, v);  // later groups were requested a step ahead (below)
        if (E.resid) asm volatile("cp.async.wait_group 0;" ::: "memory");
        if (have) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        qbar();  // residual block visible to the quadrant; the previous step's row stores have left X[step^1] and Y
        if (E.resid) {
          if (g + 1 < ngroups) issue_resid(true, b, m0, n0, g + 1, X0 + ((step + 1) & 1) * EPI_BUF);
          else issue_resid(more, nb, nm0, nn0, 0, X0 + ((step + 1) & 1) * EPI_BUF);
        }
        float x[16];
        if (have) {  // warp-uniform: tcgen05.ld is .sync.aligned
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = __uint_as_float(v[i]);
          if (c0 + 64 < p.bn && n + 64 < p.N) tmem_ld16(tacc + (uint32_t)(c0 + 64), v);  // next group's accumulator chunk: in flight during the math
        }
        if (have && row_ok) {
          const int ch = n % E.cmod;
          if (E.bias) {
            float bv[16];
            ldg16(E.bias + ch, bv);
#pragma unroll
            for (int i = 0; i < 16; ++i) x[i] += bv[i];
          }
          uint32_t xp[8];
          round16(x, xp);  // the reference's layer output is bf16
          if (E.scale) {
            float sv[16];
            ldg16(E.scale + ch, sv);
#pragma unroll
            for (int i = 0; i < 16; ++i) x[i] *= sv[i];
            round16(x, xp);
          }
          if (E.resid) {
            const uint4 r0 = lds128(Xc + own0), r1 = lds128(Xc + own1);
            const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) { x[2 * i] += bf16lo(rr[i]); x[2 * i + 1] += bf16hi(rr[i]); }
            round16(x, xp);
          }
          if (E.out_raw) {
            sts128(Xc + own0, make_uint4(xp[0], xp[1], xp[2], xp[3]));
            sts128(Xc + own1, make_uint4(xp[4], xp[5], xp[6], xp[7]));
          }
          if (E.out_act) {
            float y[16];
            if constexpr (ACT == ACT_SNAKE) {
              float ea[16], ib[16];
              ldg16(E.snake_ea + ch, ea);
              ldg16(E.snake_ib + ch, ib);
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float sn = snake_sin(x[i] * ea[i]);
                y[i] = x[i] + ib[i] * sn * sn;
              }
            } else if constexpr (ACT == ACT_GELU) {
#pragma unroll
              for (int i = 0; i < 16; ++i) y[i] = gelu_erf(x[i]);
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) y[i] = x[i];
            }
            uint4 o0, o1;
            o0.x = pack_bf16(y[0], y[1]); o0.y = pack_bf16(y[2], y[3]); o0.z = pack_bf16(y[4], y[5]); o0.w = pack_bf16(y[6], y[7]);
            o1.x = pack_bf16(y[8], y[9]); o1.y = pack_bf16(y[10], y[11]); o1.z = pack_bf16(y[12], y[13]); o1.w = pack_bf16(y[14], y[15]);
            sts128(Y + own0, o0);
            sts128(Y + own1, o1);
          }
        }
        qbar();  // the quadrant's block is complete in shared memory
        if (E.out_raw) store_rows(Xc, E.out_raw, p.raw_bs, b, m0, n0, g);
        if (E.out_act) store_rows(Y, E.out_act, p.act_bs, b, m0, n0, g);
      }
    }
    // this warp has read its part of the accumulator: hand it back to the MMA issuer (one arrival per epilogue warp)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tempty0 + 8 * acc) : "memory");
    }  // tile loop
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * acc_cols) : "memory");
  }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn g_encode = nullptr;
int g_sm_count = 0;

}  // namespace

int gemm_init() {
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    Q3_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    Q3_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available in this driver");
    g_encode = reinterpret_cast<EncodeFn>(fn);
  }
  Q3_CUDA(cudaFuncSetAttribute(tap_gemm_kernel<ACT_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_OPTIN));
  Q3_CUDA(cudaFuncSetAttribute(tap_gemm_kernel<ACT_SNAKE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_OPTIN));
  Q3_CUDA(cudaFuncSetAttribute(tap_gemm_kernel<ACT_GELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_OPTIN));
  Q3_CUDA(cudaFuncSetAttribute(tap_gemm_kernel<ACT_SWIGLU_PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_OPTIN));
  Q3_CUDA(cudaFuncSetAttribute(tap_gemm_kernel<ACT_SWIGLU_BLK8>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_OPTIN));
  if (g_sm_count == 0) {
    int dev = 0;
    Q3_CUDA(cudaGetDevice(&dev));
    Q3_CUDA(cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev));
  }
  return 0;
}

int gemm_make_plan(GemmPlan* plan, const bf16* a, int B, int T, int K, int64_t lda, int64_t a_batch_stride, const bf16* w,
                   int N, int Kp, int ntaps, const int* shifts, int bn, const GemmEpilogue& ep) {
  return gemm_make_plan_v(plan, a, B, T, K, lda, a_batch_stride, w, N, Kp, ntaps, shifts, bn, ep, GemmViews{});
}

int gemm_make_plan_v(GemmPlan* plan, const bf16* a, int B, int T, int K, int64_t lda, int64_t a_batch_stride, const bf16* w,
                     int N, int Kp, int ntaps, const int* shifts, int bn, const GemmEpilogue& ep, const GemmViews& v) {
  Q3_REQUIRE(g_encode, "gemm_init() not called");
  Q3_REQUIRE(Kp % BK == 0 && Kp >= K, "Kp must be a multiple of 64 and >= K");
  Q3_REQUIRE(bn % 16 == 0 && bn >= 16 && bn <= 256, "bn must be a multiple of 16 in [16,256]");
  Q3_REQUIRE(N % 16 == 0, "N must be a multiple of 16");
  Q3_REQUIRE(ntaps >= 1 && ntaps <= 8, "ntaps out of range");
  Q3_REQUIRE(ep.cmod % 16 == 0 && ((uintptr_t)ep.bias % 16) == 0 && ((uintptr_t)ep.scale % 16) == 0 &&
                 ((uintptr_t)ep.snake_ea % 16) == 0 && ((uintptr_t)ep.snake_ib % 16) == 0,
             "per-channel epilogue vectors must be 16-byte aligned and the channel count a multiple of 16");
  Q3_REQUIRE(!((ep.act == ACT_SWIGLU_PAIR || ep.act == ACT_SWIGLU_BLK8) && (ep.resid || ep.out_raw || ep.scale)),
             "gated epilogues write out_act only");
  Q3_REQUIRE((lda * 2) % 16 == 0 && (a_batch_stride * 2) % 16 == 0 && ((uintptr_t)a % 16) == 0, "A alignment");
  memset(plan, 0, sizeof(*plan));
  plan->B = B; plan->T = T; plan->N = N; plan->Kp = Kp; plan->ntaps = ntaps; plan->bn = bn; plan->ep = ep;
  const bool half = ep.act == ACT_SWIGLU_PAIR || ep.act == ACT_SWIGLU_BLK8;
  plan->a_row0 = v.a_row0;
  plan->nst = stages_for(bn);
  plan->raw_bs = v.raw_bs ? v.raw_bs : (long long)T * N;
  plan->act_bs = v.act_bs ? v.act_bs : (long long)T * (half ? N / 2 : N);
  plan->resid_bs = v.resid_bs ? v.resid_bs : (long long)T * N;
  const int a_rows = v.a_rows ? v.a_rows : T;
  for (int i = 0; i < ntaps; ++i) plan->shift[i] = shifts[i];
  {
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)a_rows, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)lda * 2, (cuuint64_t)a_batch_stride * 2};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)BM, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = g_encode(&plan->tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void*)a, dims, strides, box, es,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    Q3_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(A) failed: %d (K=%d T=%d B=%d lda=%lld)", (int)r, K, T, B, (long long)lda);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)ntaps * Kp, (cuuint64_t)N};
    cuuint64_t strides[1] = {(cuuint64_t)ntaps * Kp * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)bn};
    cuuint32_t es[2] = {1, 1};
    CUresult r = g_encode(&plan->tmW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)w, dims, strides, box, es,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    Q3_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(W) failed: %d (N=%d Kp=%d taps=%d)", (int)r, N, Kp, ntaps);
  }
  return 0;
}

int gemm_pick_bn(int N, int mtiles, int B) {
  static const int cand[] = {256, 240, 224, 208, 192, 176, 160, 144, 128, 112, 96, 80, 64};
  int best_small = 0;
  for (int bn : cand) {
    if (N % bn) continue;
    if ((long long)mtiles * (N / bn) * B >= 148) return bn;
    best_small = bn;
  }
  if (best_small) return best_small;
  for (int bn : cand)
    if (bn <= N) return bn;
  return N;  // N < 64 (multiple of 16)
}

int gemm_launch(const GemmPlan& plan, cudaStream_t stream, int max_ctas) {
  const long long total = (long long)((plan.T + BM - 1) / BM) * ((plan.N + plan.bn - 1) / plan.bn) * plan.B;
  int ctas = g_sm_count > 0 ? g_sm_count : 148;  // persistent: one CTA per SM walks the tiles
  if (max_ctas > 0) ctas = std::min(ctas, max_ctas);
  const int grid = (int)std::min<long long>(total, ctas);
  static const bool trace = getenv("Q3_GEMM_TRACE") != nullptr;  // tools/codec_breakdown.py joins this with an ncu launch list
  if (trace)
    fprintf(stderr, "[tap_gemm] B=%d T=%d N=%d Kp=%d taps=%d bn=%d tiles=%lld act=%d resid=%d\n", plan.B, plan.T, plan.N, plan.Kp,
            plan.ntaps, plan.bn, total, plan.ep.act, plan.ep.resid ? 1 : 0);
  const int smem_bytes = 1024 + plan.nst * stage_bytes_for(plan.bn) + BAR_BYTES + EPI_BYTES;
  switch (plan.ep.act) {
    case ACT_NONE: tap_gemm_kernel<ACT_NONE><<<grid, GEMM_THREADS, smem_bytes, stream>>>(plan); break;
    case ACT_SNAKE: tap_gemm_kernel<ACT_SNAKE><<<grid, GEMM_THREADS, smem_bytes, stream>>>(plan); break;
    case ACT_GELU: tap_gemm_kernel<ACT_GELU><<<grid, GEMM_THREADS, smem_bytes, stream>>>(plan); break;
    case ACT_SWIGLU_PAIR: tap_gemm_kernel<ACT_SWIGLU_PAIR><<<grid, GEMM_THREADS, smem_bytes, stream>>>(plan); break;
    case ACT_SWIGLU_BLK8: tap_gemm_kernel<ACT_SWIGLU_BLK8><<<grid, GEMM_THREADS, smem_bytes, stream>>>(plan); break;
    default: Q3_REQUIRE(false, "unknown activation %d", plan.ep.act);
  }
  Q3_CUDA(cudaGetLastError());
  return 0;
}

#include "../../include/qwen3tts_b200.h"

// Test hook: one tap-GEMM launch through the production planning (gemm_make_plan_v, gemm_pick_bn) and launch path.  The
// checks here cover only what the kernel would otherwise dereference blindly; gemm_make_plan_v refuses the rest.
extern "C" int q3_debug_tap_gemm(const q3_tap_gemm_desc* d, void* stream) {
  Q3_REQUIRE(d && d->a && d->w, "tap_gemm: null descriptor, A or W");
  Q3_REQUIRE(d->B >= 1 && d->T >= 1 && d->K >= 1 && d->N >= 1, "tap_gemm: empty problem (B=%d T=%d K=%d N=%d)", d->B, d->T, d->K, d->N);
  Q3_REQUIRE(d->act >= ACT_NONE && d->act <= ACT_SWIGLU_BLK8, "tap_gemm: unknown activation %d", d->act);
  Q3_REQUIRE(d->bn >= 0 && d->max_ctas >= 0 && d->cmod >= 0 && d->a_rows >= 0 && d->a_row0 >= 0, "tap_gemm: negative field");
  const bool gated = d->act == ACT_SWIGLU_PAIR || d->act == ACT_SWIGLU_BLK8;
  Q3_REQUIRE(d->out_raw || d->out_act, "tap_gemm: no output");
  Q3_REQUIRE(!gated || d->out_act, "tap_gemm: gated epilogues need out_act");
  Q3_REQUIRE(d->act != ACT_SNAKE || !d->out_act || (d->snake_ea && d->snake_ib), "tap_gemm: SnakeBeta needs snake_ea and snake_ib");
  // every store and residual load moves 16 bytes: outputs / residual and their batch strides must keep that alignment
  Q3_REQUIRE((uintptr_t)d->out_raw % 16 == 0 && (uintptr_t)d->out_act % 16 == 0 && (uintptr_t)d->resid % 16 == 0 &&
                 d->raw_bs % 8 == 0 && d->act_bs % 8 == 0 && d->resid_bs % 8 == 0,
             "tap_gemm: outputs / residual must be 16-byte aligned with batch strides that are multiples of 8 elements");
  if (gemm_init()) return 1;
  GemmEpilogue ep{};
  ep.bias = d->bias; ep.scale = d->scale; ep.resid = reinterpret_cast<const bf16*>(d->resid);
  ep.snake_ea = d->snake_ea; ep.snake_ib = d->snake_ib;
  ep.cmod = d->cmod ? d->cmod : d->N;
  ep.act = d->act;
  ep.out_raw = reinterpret_cast<bf16*>(d->out_raw); ep.out_act = reinterpret_cast<bf16*>(d->out_act);
  GemmViews v;
  v.a_rows = d->a_rows; v.a_row0 = d->a_row0;
  v.raw_bs = d->raw_bs; v.act_bs = d->act_bs; v.resid_bs = d->resid_bs;
  const int a_rows = d->a_rows ? d->a_rows : d->T;
  const int64_t a_bs = d->a_bs ? d->a_bs : (int64_t)a_rows * d->K;
  const int bn = d->bn ? d->bn : gemm_pick_bn(d->N, (d->T + BM - 1) / BM, d->B);
  GemmPlan plan;
  if (gemm_make_plan_v(&plan, reinterpret_cast<const bf16*>(d->a), d->B, d->T, d->K, d->K, a_bs, reinterpret_cast<const bf16*>(d->w),
                       d->N, d->Kp, d->ntaps, d->shifts, bn, ep, v))
    return 1;
  return gemm_launch(plan, reinterpret_cast<cudaStream_t>(stream), d->max_ctas);
}
