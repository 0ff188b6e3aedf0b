// Constant-Q projection on the tensor cores: per octave the 172 x 256 x 72 contraction
//   C[(b,t)][n] = sum_k xpad_o[b][t*hop_o + k] * W[k][n]          (n interleaves real / imaginary parts of 36 bins)
// as tcgen05.mma kind::f16 on a three-way bf16 split of both operands (x = hi + mid + lo, each round-to-nearest bf16;
// the six products hi*hi, hi*mid, mid*hi, hi*lo, lo*hi, mid*mid are accumulated in FP32 in TMEM; the dropped terms are
// below 2^-24 of |a||w|).  A single bf16 / TF32 product is far from the 1e-3 bar for this stage and even a two-way
// split leaves ~1e-3 in the weak bins of the log spectrum (SURVEY.md F6 / Appendix C.4; measured here with 3xTF32);
// the three-way split reproduces FP32-class results.
//
// Replaces (together with the unchanged decimation chain) reference: basic_pitch/layers/nnaudio.py:216-256
// (`get_cqt_complex`, reflect pad + two strided conv1d per octave), :642-661 (concat, sqrt(len) scaling, magnitude) and
// layers/signal.py:174-176 (power -> 10*log10(. + 1e-10)); the per-window min / max feed lognorm_kernel (hcqt.cu).
//
// The A operand is an overlapping strided view of the signal (row t starts at sample t*hop), which no UMMA/TMA
// descriptor can express for hop*4 B < 16 B or non-canonical pitches, so producer warps build it explicitly (reflect
// padding and three-way split included) and write it to TENSOR memory, where TS-form MMAs read it.  A producer lane owns
// one frame row: it loads its 16 taps of the chunk (global memory through L1: the rows of an item overlap, the lines stay
// hot), splits them three ways in registers and writes them with tcgen05.st straight into the tensor-memory columns the
// MMAs read (kind::f16 A-in-TMEM layout: row = lane, two bf16 per column, K = 16 -> 8 columns; 3 planes x 32 columns per
// chunk).  No operand tile in shared memory, so the whole split kernel matrix (120 KB) stays resident instead of being
// streamed per chunk.  Shared-memory traffic per chunk: 60 KB of B reads.
//
// item = (M-tile of 128 frames, octave); per item 4 K-chunks of 64 taps, each chunk = 4 k-steps x 6 products:
//   warps 8-23  producers: warp w serves TMEM lane quadrant w % 4 and the taps 16 (w / 4) .. 16 (w / 4) + 15 of every
//               chunk (k-step w / 4); tcgen05.st of the three planes, mbarrier arrive
//   warp 24     MMA issuer (one elected lane): bulk-copies the split kernel matrix once per CTA, then 24 TS-form
//               tcgen05.mma per chunk; tcgen05.commit frees the A stage / publishes the accumulator
//   warps 0-7   epilogue (two per TMEM lane quadrant): tcgen05.ld 32 / 40 columns, magnitude * sqrt(len), log-power, store,
//               per-window min/max (atomics)
// (the warp scheduler prefers high warp ids when it picks the next instruction: the MMA issuer and the producers
// outrank the epilogue)
// Shared memory: the split kernel matrix + the epilogue's staging tiles; tensor memory: 3 A stages x 96 columns at
// 0 / 96 / 192, accumulators (80 columns) at 288 and 416.
#include <cuda_bf16.h>

#include <cstdio>
#include <cstdlib>
#include <vector>

#include "kernels.cuh"
#include "tc_ptx.cuh"

namespace bp {

namespace cq {
constexpr int kMTile = 128;
constexpr int kKc = 64;                          // taps per chunk
constexpr int kN = 80;                           // 72 columns padded to a multiple of 16
constexpr int kWPlane = (kKc / 8) * kN * 16;      // 10240 B : [8 k-chunks of 8][80][16 B]
constexpr int kWBytes = 4 * 3 * kWPlane;          // 122 880: the whole split kernel matrix
constexpr int kProducers = 4 * (kKc / 16) * 32;   // 4 TMEM lane quadrants x 4 k-steps x 32 lanes (rows): 16 producer warps
static_assert(kProducers == 512, "producer geometry");
constexpr int kEpiWarps = 8;                      // two per TMEM lane quadrant: bins 0..15 / 16..35 of the octave
constexpr int kThreads = kProducers + 32 + 32 * kEpiWarps;
static_assert(kThreads <= 1024, "block size");
constexpr int kTilePitch = 21;                    // epilogue staging: [8 warps][32 rows][<= 20 bins + 1]
constexpr int kEpiBytes = kEpiWarps * 32 * kTilePitch * 4;
constexpr int kSmemBytes = kWBytes + kEpiBytes + 256;
// tensor memory (512 columns)
constexpr int kStages = 3;                        // A operand stages
constexpr int kAStageCols = 96;
constexpr int kAccCol0 = 288, kAccCol1 = 416;  // (+32 stays a multiple of 32 for the epilogue's x32 loads)
}  // namespace cq


static inline uint16_t f2bf_rn(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline float bf2f_(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// kernel matrix, three-way bf16 split, laid out per chunk: wtc[chunk 4][plane 3][k/8 8][n 80][8] (bf16)
void build_cqt_tc_weights(const float* cqt_real /* [36][256] */, const float* cqt_imag, std::vector<uint16_t>& out) {
  out.assign((size_t)4 * 3 * 8 * cq::kN * 8, 0);
  for (int k = 0; k < kTaps; ++k)
    for (int n = 0; n < 72; ++n) {
      const float w = (n & 1) ? cqt_imag[(n >> 1) * kTaps + k] : cqt_real[(n >> 1) * kTaps + k];
      const uint16_t h = f2bf_rn(w);
      const float r1 = w - bf2f_(h);
      const uint16_t m = f2bf_rn(r1);
      const uint16_t l = f2bf_rn(r1 - bf2f_(m));
      const int c = k / cq::kKc, kk = k % cq::kKc;
      const size_t plane = (size_t)8 * cq::kN * 8;
      const size_t base = (size_t)c * 3 * plane;
      const size_t off = ((size_t)(kk >> 3) * cq::kN + n) * 8 + (kk & 7);
      out[base + off] = h;
      out[base + plane + off] = m;
      out[base + 2 * plane + off] = l;
    }
}

struct CqtTcArgs {
  const float* audio;
  const WinDesc* desc;   // may be null: window b = audio + b*43844
  const float* chain;    // decimated signals x_1..x_8
  const uint16_t* wtc;   // split kernel matrix (bf16), 4 chunks of 30 KB
  const float* scale;    // [309] sqrt(kernel length)
  float* logmag;         // [B][172][309]
  unsigned int* minmax;  // [B][2] ordered-uint min / max
  int n_windows, n_mtiles;
  long long* trace;  // -DBP_TC_TRACE: [item][16] clock64 stamps of CTA 0
};

#ifdef BP_TC_TRACE
#define CQ_TRACE(i, ev) do { if (a.trace && blockIdx.x == 0 && (i) < 64 && (threadIdx.x & 31) == 0) a.trace[(i) * 16 + (ev)] = clock64(); } while (0)
#else
#define CQ_TRACE(i, ev) do { } while (0)
#endif

__global__ void __launch_bounds__(cq::kThreads, 1) cqt_ts_kernel(const CqtTcArgs a) {
  using namespace cq;
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* s_w = smem;  // [chunk 4][plane 3][k/8 8][n 80][16 B]
  float* s_tile = reinterpret_cast<float*>(smem + kWBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWBytes + kEpiBytes);
  uint64_t* a_full = bars;                  // [3] 16 producer-warp arrivals
  uint64_t* a_empty = bars + kStages;       // [3] commit behind the MMAs that read the stage
  uint64_t* tmem_full = a_empty + kStages;  // [2]
  uint64_t* tmem_empty = tmem_full + 2;     // [2]
  uint64_t* w_full = tmem_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // broadcast: warp-uniform role branches and loop state
  const int lane = threadIdx.x & 31;
  constexpr int kMmaWarp = kEpiWarps + kProducers / 32;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(a_full + s, kProducers / 32);
      mbar_init(a_empty + s, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tmem_full + i, 1);
      mbar_init(tmem_empty + i, kEpiWarps);
    }
    mbar_init(w_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_items = a.n_mtiles * kOctaves;
  const int total_frames = a.n_windows * kFrames;

  if (warp >= kEpiWarps && warp < kMmaWarp) {
    // ------------------------------ producers ------------------------------
    const int pw = warp - kEpiWarps;
    const int quad = pw & 3, ks = pw >> 2;  // TMEM lane quadrant; k-step (taps 16 ks .. 16 ks + 15 of every chunk)
    const int row = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    uint32_t g = 0;  // chunks produced so far -> stage g % 3
    int icnt = -1;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      ++icnt;
      if (pw == 0) CQ_TRACE(icnt, 0);  // producer warp 0 starts the item
      const int mt = it / kOctaves, o = it % kOctaves;
      const int hop = 256 >> o;
      const int len = octave_len_rt(o);
      const int m = mt * kMTile + row;
      const bool live = m < total_frames;
      const int b = live ? m / kFrames : 0;
      const int t = m - b * kFrames;
      const float* src;
      int lo = 0, hi = len;
      if (o == 0) {
        if (a.desc) {
          const WinDesc d = a.desc[b];
          src = a.audio + d.base;
          lo = d.lo;
          hi = d.hi;
        } else {
          src = a.audio + (long long)b * kWinSamples;
        }
      } else {
        src = a.chain + (size_t)b * kChainStride + chain_off_rt(o);
      }
      const int i0 = t * hop - 128 + 16 * ks;  // signal index of this lane's first tap in chunk 0
      auto load16 = [&](int c, float (&x)[16]) {
        const int ib = i0 + c * kKc;
        if (live && ib >= max(lo, 0) && ib + 16 <= min(hi, len) && ((reinterpret_cast<uintptr_t>(src + ib) & 15) == 0)) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(src + ib) + q);
            x[4 * q] = v.x, x[4 * q + 1] = v.y, x[4 * q + 2] = v.z, x[4 * q + 3] = v.w;
          }
        } else {
          // rows at the signal ends (reflect padding, zeros outside [lo, hi)), unaligned low octaves, dead rows
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            int idx = ib + k;
            if (idx < 0) idx = -idx;
            if (idx >= len) idx = 2 * (len - 1) - idx;
            x[k] = (live && idx >= lo && idx < hi) ? __ldg(src + idx) : 0.f;
          }
        }
      };
      float xn[16];
      load16(0, xn);
      for (int c = 0; c < kTaps / kKc; ++c, ++g) {
        float x[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) x[k] = xn[k];
        if (c + 1 < kTaps / kKc) load16(c + 1, xn);  // the next chunk's loads are in flight while this one is split and stored
        uint32_t h[8], md[8], l[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const __nv_bfloat162 hh = __floats2bfloat162_rn(x[2 * j], x[2 * j + 1]);
          const float2 hf = __bfloat1622float2(hh);
          const float r0 = x[2 * j] - hf.x, r1 = x[2 * j + 1] - hf.y;
          const __nv_bfloat162 mm = __floats2bfloat162_rn(r0, r1);
          const float2 mf = __bfloat1622float2(mm);
          const __nv_bfloat162 ll = __floats2bfloat162_rn(r0 - mf.x, r1 - mf.y);
          h[j] = *reinterpret_cast<const uint32_t*>(&hh);
          md[j] = *reinterpret_cast<const uint32_t*>(&mm);
          l[j] = *reinterpret_cast<const uint32_t*>(&ll);
        }
        const uint32_t stage = g % kStages, ph = (g / kStages) & 1u;
        if (pw == 0) CQ_TRACE(icnt, 14 + (c & 1));  // (c = 2, 3 overwrite: last split done)
        mbar_wait(a_empty + stage, ph ^ 1u);
        if (pw == 0) CQ_TRACE(icnt, 2 + c);  // stage acquired for chunk c
        tc_fence_after();
        const uint32_t col = lane_base + stage * kAStageCols + (uint32_t)ks * 8u;
        tmem_st8(col, h);
        tmem_st8(col + 32, md);
        tmem_st8(col + 64, l);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full + stage);
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------ MMA issuer (A operand in tensor memory) ------------------------------
    constexpr uint32_t idesc = make_idesc(128, kN);
    const uint32_t leader = elect_one() ? 1u : 0u;
    // the whole split kernel matrix, once per CTA
    bulk_g2s_expect_pred(s_w, a.wtc, kWBytes, w_full, leader);
    const uint32_t desc_hi32 = (128u >> 4) | (1u << 14);
    const uint32_t w_base = ((smem_u32(s_w) >> 4) & 0x3fffu) | ((uint32_t)(kN * 16 >> 4) << 16);
    uint32_t g = 0, icount = 0;
    uint32_t ph_t[2] = {0, 0};
    mbar_wait(w_full, 0);
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      const uint32_t buf = icount & 1u;
      mbar_wait(tmem_empty + buf, ph_t[buf] ^ 1);
      ph_t[buf] ^= 1;
      tc_fence_after();
      const uint32_t d = tmem_base + (buf ? kAccCol1 : kAccCol0);
      CQ_TRACE(icount, 6);  // accumulator acquired
      for (int c = 0; c < kTaps / kKc; ++c, ++g) {
        const uint32_t stage = g % kStages, ph = (g / kStages) & 1u;
        mbar_wait(a_full + stage, ph);
        CQ_TRACE(icount, 7 + c);  // chunk c's operands arrived
        tc_fence_after();
        const uint32_t acol = tmem_base + stage * kAStageCols;
#pragma unroll
        for (int ks = 0; ks < kKc / 16; ++ks) {
          const uint32_t ah = acol + (uint32_t)ks * 8u;
          const uint32_t bo = w_base + (uint32_t)(((c * 3) * (kWPlane) + ks * 2 * (kN * 16)) >> 4);
          umma_ts_bf16_x6(d, ah, ah + 32u, ah + 64u, bo, bo + (kWPlane >> 4), bo + 2 * (kWPlane >> 4), desc_hi32, idesc,
                          (c | ks) ? 1u : 0u, leader);
        }
        umma_commit_pred(a_empty + stage, leader);
      }
      umma_commit_pred(tmem_full + buf, leader);
      CQ_TRACE(icount, 11);  // all MMAs of the item issued
      ++icount;
    }
  } else {
    // ------------------------------ epilogue (warps 0..7) ------------------------------
    // Two warps per TMEM lane quadrant (a warp may only read lanes 32 (warp % 4) ..): warp < 4 takes bins 0..15 of the
    // octave (accumulator columns 0..31), warp >= 4 bins 16..35 (columns 32..71).  Four warps alone were the bottleneck
    // of the kernel (busy all the time while the tensor pipe idled).
    const int quad = warp & 3, half = warp >> 2;
    const int row = quad * 32 + lane;
    const int nb = half ? 20 : 16, bin0 = half ? 16 : 0;
    uint32_t ph_t[2] = {0, 0};
    uint32_t icount = 0;
    float* tile = s_tile + warp * (32 * kTilePitch);
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      const int mt = it / kOctaves, o = it % kOctaves;
      const int m = mt * kMTile + row;
      const bool live = m < total_frames;
      const int b = live ? m / kFrames : -1;
      const uint32_t buf = icount & 1u;
      mbar_wait(tmem_full + buf, ph_t[buf]);
      ph_t[buf] ^= 1;
      tc_fence_after();
      if (warp == 0) CQ_TRACE(icount, 12);  // epilogue saw the accumulator
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (buf ? kAccCol1 : kAccCol0) + (uint32_t)(2 * bin0);
      float vmin = INFINITY, vmax = -INFINITY;
      const int g0 = (8 - o) * kBinsPerOctave - 15 + bin0;  // global bin of this warp's first bin (negative for the lowest of o = 8)
      // 10*log10(re^2 + im^2 + 1e-10) per bin (MUFU.LG2; the reference's sqrt-then-square differs by < 1e-6 dB), staged
      // per warp in shared memory so that the stores below write runs of consecutive bins instead of one bin of 32 rows
      uint32_t v[40];
      tmem_ld32_nowait(taddr, reinterpret_cast<uint32_t(&)[32]>(v[0]));
      if (half) {
        uint32_t t8[8];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(t8[0]), "=r"(t8[1]), "=r"(t8[2]), "=r"(t8[3]), "=r"(t8[4]), "=r"(t8[5]), "=r"(t8[6]), "=r"(t8[7])
                     : "r"(taddr + 32));
#pragma unroll
        for (int k = 0; k < 8; ++k) v[32 + k] = t8[k];
      }
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty + buf);  // the accumulator is free: the values are in registers
#pragma unroll
      for (int j = 0; j < 20; ++j) {
        if (j < nb) {
          const int g = g0 + j;
          float L = 0.f;
          if (g >= 0) {
            const float s = __ldg(a.scale + g);
            const float re = __uint_as_float(v[2 * j]) * s, im = __uint_as_float(v[2 * j + 1]) * s;
            L = __log2f(fmaf(re, re, im * im) + 1e-10f) * 3.0102999566398120f;
            if (live) {
              vmin = fminf(vmin, L);
              vmax = fmaxf(vmax, L);
            }
          }
          tile[lane * kTilePitch + j] = L;
        }
      }
      __syncwarp();
      {
        const int m0 = mt * kMTile + quad * 32;
        int rr = half ? lane / 20 : lane >> 4, jj = half ? lane - 20 * rr : lane & 15;
        for (int i = 0; i < nb; ++i) {  // 32 rows x nb bins, consecutive lanes -> consecutive bins of a row
          if (m0 + rr < total_frames && g0 + jj >= 0) a.logmag[(size_t)(m0 + rr) * kCqtBins + g0 + jj] = tile[rr * kTilePitch + jj];
          jj += 32;  // the next element this lane owns is 32 further: one or two rows down
          if (half) {
            rr += 1 + (jj >= 40);
            jj -= jj >= 40 ? 40 : 20;
          } else {
            rr += 2;
            jj -= 32;
          }
        }
      }
      __syncwarp();  // the staging tile is reused by the next item
      // per-window min / max: one atomic pair per warp when the whole warp sits in one window
      const int b0 = __shfl_sync(0xffffffffu, b, 0);
      const bool uniform = __all_sync(0xffffffffu, b == b0);
      if (uniform) {
        if (b0 >= 0) {
#pragma unroll
          for (int off = 16; off; off >>= 1) {
            vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, off));
            vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, off));
          }
          if (lane == 0 && vmin <= vmax) {
            atomicMin(a.minmax + 2 * b0, float_to_ordered(vmin));
            atomicMax(a.minmax + 2 * b0 + 1, float_to_ordered(vmax));
          }
        }
      } else if (live && vmin <= vmax) {
        atomicMin(a.minmax + 2 * b, float_to_ordered(vmin));
        atomicMax(a.minmax + 2 * b + 1, float_to_ordered(vmax));
      }
      if (warp == 0) CQ_TRACE(icount, 13);  // epilogue done
      ++icount;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

__global__ void minmax_init_kernel2(unsigned int* mm, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    mm[2 * i] = 0xffffffffu;
    mm[2 * i + 1] = 0u;
  }
}

void cqt_tc_setup() {
  cudaFuncSetAttribute(cqt_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cq::kSmemBytes);
}

void launch_cqt_tc(const float* audio, const WinDesc* desc, const float* chain, const uint16_t* wtc, const float* scale,
                   float* logmag, unsigned int* minmax, int n_windows, int n_sms, cudaStream_t st) {
  minmax_init_kernel2<<<(n_windows + 255) / 256, 256, 0, st>>>(minmax, n_windows);
  CqtTcArgs a;
  a.trace = nullptr;
#ifdef BP_TC_TRACE
  static long long* d_trace = nullptr;
  const bool tracing = getenv("BP_TC_TRACE") != nullptr;
  if (tracing) {
    if (!d_trace) cudaMalloc(&d_trace, 64 * 16 * sizeof(long long));
    cudaMemsetAsync(d_trace, 0, 64 * 16 * sizeof(long long), st);
    a.trace = d_trace;
  }
#endif
  a.audio = audio;
  a.desc = desc;
  a.chain = chain;
  a.wtc = wtc;
  a.scale = scale;
  a.logmag = logmag;
  a.minmax = minmax;
  a.n_windows = n_windows;
  a.n_mtiles = (n_windows * kFrames + cq::kMTile - 1) / cq::kMTile;
  const int n_items = a.n_mtiles * kOctaves;
  const int grid = n_items < n_sms ? n_items : n_sms;
  cqt_ts_kernel<<<grid, cq::kThreads, cq::kSmemBytes, st>>>(a);
#ifdef BP_TC_TRACE
  if (tracing) {
    static long long h[64 * 16];
    cudaMemcpyAsync(h, d_trace, sizeof(h), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    fprintf(stderr, "cqt_trace n_items %d grid %d (columns: 0 item start, 1 unused, 2-5 stage acquired c0..c3, 6 acc acquired, 7-10 operands arrived c0..c3, 11 MMAs issued, 12 epilogue saw, 13 epilogue done, 14-15 split done c2, c3)\n", n_items, grid);
    for (int i = 0; i < 64 && h[i * 16]; ++i) {
      fprintf(stderr, "item %2d (octave %d):", i, (i * grid) % 9);
      for (int e = 0; e < 16; ++e) fprintf(stderr, " %7lld", h[i * 16 + e] ? h[i * 16 + e] - h[0] : -1);
      fprintf(stderr, "\n");
    }
  }
#endif
}

}  // namespace bp
