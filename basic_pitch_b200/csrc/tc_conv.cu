// The three wide convolutions — contour (8 -> 8 channels, 3 x 39 taps, 65 % of the model's FLOPs), onset
// (8 -> 32 channels, 5 x 5 taps, frequency stride 3, 18 %) and note (1 -> 32 channels, 7 x 7, stride 3, 4.5 %) —
// on the 5th-gen tensor cores: tcgen05.mma (kind::f16, bf16 operands, fp32 accumulators in TMEM), operands staged in shared
// memory by bulk async copies (UBLKCP) signalled through mbarriers, warp-specialised roles.
//
// Replaces nodes 231/232 (contour conv + ReLU, reference: basic_pitch/models.py:241-250) and 230/243 (onset
// conv + ReLU, reference: basic_pitch/models.py:295-304) of the deployed graph, and the harmonic stacking in
// front of them (reference: basic_pitch/nn.py:69-88), which is folded into the weight operand and never
// materialised; node 238/239 (note conv1 + ReLU, models.py:270-279) reads the contour posteriorgram instead.
// One kernel template, three specs (TcConvSpec).  The epilogue (EPI 1 / 2 / 3 = onset / note / contour) also computes
// the FOLLOWING single-output convolution (onset conv2 models.py:305-313, note conv2 :282-290, contour conv2 :254-262)
// completely, so neither the 8- / 32-channel activations nor any partial sums of them reach HBM:
//   * channels and frequency taps are reduced by a SECOND tensor-core contraction whose A operand is bias + ReLU of the
//     accumulator, split to bf16 hi/lo and written back into the same tensor-memory columns (TS-form MMAs, see TcB2),
//   * the time taps are summed across the lanes of the warp (the 32 lanes hold 32 consecutive frames: shuffles) and
//     across the four epilogue warps of an accumulator slot through a small shared-memory exchange; M-tiles overlap
//     by KH2 - 1 rows, so every frame is complete in exactly one tile.  The thread of tile row r finishes the output
//     frame r - H (H = KH2 / 2), so every tap comes from a lane at or below its own: each lane adds its taps in the
//     same order whatever its position in the tile, and a frame's value does not depend on the batch around it,
//   * the frequency halo between neighbouring tiles is a register carry: a slot walks its frequency tiles in ascending
//     order; only where two tile RANGES meet (slot 0 | slot 1, or the group splits of a small batch) the two partial
//     sums go to a small edge buffer and edge_fix_kernel finishes those 4 (contour) / 2 bins,
//   * bias, sigmoid (+ the note input channel of the onset conv2, + unwrap inference.py:247-279) and the store.
// EPI 0 stores the contour activations channels-last (path 2, activation-level tests).
//
// Formulation ("Toeplitz along frequency on aligned chunks")
//   rows  m = b*174 + t            time frames of all windows of the chunk, two zero rows between windows
//   D[m][(fl,co)] (+)= A[m+dt][8c .. 8c+15] x T(dt,off)[16][(fl,co)]
//     A      the normalised CQT y itself (NOT the 8-channel stack), rows shifted by the time tap dt; K = 16 bins that
//            start on an 8-bin chunk of the k-chunk-major layout
//     T      16 x 128 "weight tile": T[k][(fl,co)] = sum_ci W[co][ci][dt][df_ci] with
//            df_ci = (8c + k) - shift_ci - SF*(ft*FLT + fl) + PL   (terms outside 0 <= df < KW or outside the stacked
//            image 0 <= g < 264 dropped).  The harmonic channels are shifted views of one image, so they are MERGED
//            in the weight operand: the stack conv is a single-channel conv of y whose taps are the union of the
//            shifted per-channel taps (contour: 8 x 39 = 312 taps on 176 distinct offsets -> 12 instead of 32
//            K-steps per time tap and frequency tile).
//            N = FLT output bins x COUT channels = 128 (contour 16 x 8, onset / note 4 x 32); a tile depends on
//            (dt, 8c - SF*FLT*ft), so frequency tiles SF*FLT*d = 8*j bins apart share tiles (de-duplicated by
//            content)
//   every (ft, dt, c) with a non-empty tile is one K=16 MMA step of shape 128 x 128 x 16
// Precision: both operands are split x = hi + lo (bf16 each) and three products are accumulated
// (hi*hi + hi*lo + lo*hi) in fp32, which keeps the posteriorgrams within ~1e-5 of the FP32 path
// (SURVEY.md Appendix C.4); a single bf16 product would miss the 1e-3 bar.
//
// Work decomposition: item = (M-tile of 128 rows, split s of S over the frequency groups); group g = the two
// frequency tiles {g, g + G0} (two accumulator slots; shared weight tiles where their content is equal).  Tensor memory:
// three 128-column conv1 accumulator regions used as a ring + the conv2 accumulators.  A CTA (1 per SM, persistent) walks items
// i = blockIdx.x, +gridDim.x, ...:
//   warp 8      producer: bulk-copies the (128+KH-1) x 320 bf16 hi/lo data tile (k-chunk-major) once per item and
//               streams the weight tiles of each group's program (8 KB each) through a 7- / 9-stage ring
//   warps 9, 10 MMA issuers, one per accumulator slot of the group (instruction issue, not the tensor pipe, limits
//               a single issuing warp at this MMA size): program words from constant memory, descriptors are
//               base + precomputed offset, 3 x tcgen05.mma per step by one elected lane, tcgen05.commit frees the
//               weight stage / publishes the accumulators
//   warp 11     conv2 MMA issuer (A operand in tensor memory)
//   warps 0-3, 4-7  epilogue, one warpgroup-like set of 4 warps (= the 4 TMEM lane quadrants) per accumulator slot:
//               tcgen05.ld the accumulator columns, + bias, ReLU, split, tcgen05.st; then the conv2 sums as described above
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <vector>

#include "kernels.cuh"
#include "tc_ptx.cuh"

namespace bp {

namespace tc {
constexpr int kMTile = 128;
constexpr int kTileBytes = 8192;                                 // weight tile: [plane 2][kchunk 2][128][8] bf16
constexpr int kMaxSteps = 1024;                                  // program steps per layer (constant memory)
constexpr int kMaxGroups = 15;
constexpr int kThreads = 384;  // 12 warps: 2 x 4 epilogue warps, producer, 2 conv1 MMA issuers, the conv2 MMA issuer
// The issue arbiter of an SM sub-partition prefers the highest warp id, so the latency-critical single-thread roles
// (producer, MMA issuers) get the highest ids and are never starved by the epilogue warps.
constexpr int kProducerWarp = 8, kMmaWarp0 = 9, kMmaWarp1 = 10, kMma2Warp = 11;
// time-halo exchange between the four epilogue warps of a slot: [slot 2][buffer 2][warp 3][kXchgFloats] (warps 0..2 of a
// slot publish their top lanes for the warp above; the last warp has nobody to publish to)
// Shared memory is laid out per layer: the data tile, then as many weight-tile stages as fit.  The weight ring is what
// bounds the conv1 MMAs (one 8 KB tile per step, about 2 000 cycles from the request to the release of its stage, most
// steps used by one slot only = 192 tensor cycles), so every KB goes to stages: contour / onset 7, note 9.
struct TcSmem {
  int data_bytes;   // [2 planes][chunks][128 + KH - 1 rows][16 B], rounded up to 1 KB
  int xchg_floats;  // per publishing warp (contour 10 lane values x 20 offsets, note 21 x 6, onset 3 x 6)
  int b2_bytes;     // conv2 weight tiles (TcB2)
  int stages;
  __host__ __device__ constexpr int xchg_bytes() const { return 2 * 2 * 3 * xchg_floats * 4; }
  __host__ __device__ constexpr int total() const { return data_bytes + stages * kTileBytes + xchg_bytes() + b2_bytes + 512; }
};
constexpr int kMaxSmem = 232448;  // 227 KB opt-in per CTA
__host__ __device__ constexpr TcSmem tc_smem(int epi) {  // epi: 0 / 3 contour, 1 onset, 2 note
  TcSmem s{};
  const int chunks = epi == 2 ? 33 : 39, rows = kMTile + (epi == 1 ? 4 : epi == 2 ? 6 : 2);
  s.data_bytes = (2 * chunks * rows * 16 + 1023) / 1024 * 1024;
  s.xchg_floats = epi == 1 ? 32 : epi == 2 ? 128 : 200;
  s.b2_bytes = epi == 2 ? 4096 : 2048;
  s.stages = (kMaxSmem - 512 - s.data_bytes - s.xchg_bytes() - s.b2_bytes) / kTileBytes;
  return s;
}
static_assert(tc_smem(0).stages == 7 && tc_smem(1).stages == 7 && tc_smem(2).stages == 9, "weight ring depth");
constexpr int kMaxStages = 9;
// step word of a slot: [0,14) A start-address offset >> 4, [15] first MMA into that accumulator; kNoUse = the
// slot's frequency tile does not use this step's weight tile
constexpr uint32_t kUseFirstAcc = 1u << 15, kNoUse = 0xffffffffu;
// Tensor memory (512 columns): three 128-column conv1 accumulators used as a ring by the frequency tiles in program order,
// then the conv2 accumulators (per-layer widths in TcB2).
constexpr int kRegions = 3;
constexpr uint32_t kD2Base = kRegions * 128;
}  // namespace tc

// ------------------------------------------------------------------------------------------------
// Host: weight tiles + per-group programs
// ------------------------------------------------------------------------------------------------
static inline uint16_t f2bf(float x) {  // round-to-nearest-even float -> bf16 bits
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline float bf2f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

//                                      KH KW SF PT PL COUT FLT WOUT n_ci  shifts                              bins ch8 rows/win lead epi KH2 HALO G0
TcConvSpec tc_contour_spec() { return {3, 39, 1, 1, 19, 8, 16, 264, 8, {-36, 0, 36, 57, 72, 84, 93, 101}, 309, 40, 174, 3, 0, 5, 2, 9}; }
TcConvSpec tc_onset_spec() { return {5, 5, 3, 2, 1, 32, 4, 88, 8, {-36, 0, 36, 57, 72, 84, 93, 101}, 309, 40, 174, 3, 1, 3, 1, 12}; }
TcConvSpec tc_note_spec() { return {7, 7, 3, 3, 2, 32, 4, 88, 1, {0, 0, 0, 0, 0, 0, 0, 0}, 264, 34, 175, 6, 2, 7, 1, 12}; }

void TcConvPlan::build(const TcConvSpec& sp, const float* W /* [COUT][n_ci][KH][KW] */) {
  using namespace tc;
  spec = sp;
  tiles.clear();
  tile_seq.clear();
  slot_words[0].clear();
  slot_words[1].clear();
  group_step_off.clear();
  group_ft.clear();
  const int n_ft = (sp.WOUT + sp.FLT - 1) / sp.FLT;
  const int data_rows = kMTile + sp.KH - 1;
  const int lbo16 = data_rows;  // (rows * 16 B) >> 4
  // K = 16 steps start on 8-bin chunk boundaries (the k-chunk-major layout makes any chunk index a legal
  // descriptor start), so frequency tiles d apart share weight tiles when SF*FLT*d is a multiple of 8 bins; the two
  // tiles of a group are G0 apart: slot 0 walks tiles 0 .. G0-1, slot 1 tiles G0 .. n_ft-1, both in ascending order
  // (the fused epilogue carries the frequency halo of the next conv from tile to tile in registers)
  const int stride = sp.G0;

  // weight tiles are de-duplicated by content (boundary clipping makes otherwise equal keys differ and vice versa)
  std::unordered_map<uint64_t, std::vector<int>> by_hash;
  int n_keys = 0;
  std::vector<uint16_t> scratch(kTileBytes / 2);
  // The n_ci input channels are shifted views of ONE image (harmonic stacking, nn.py:69-88), so the stack conv is a
  // single-channel conv of y with the merged kernel  Wm[co][dt][u] = sum_ci W[co][ci][dt][u - shift_ci + PL]  wherever
  // the stacked pixel exists (0 <= g = u_abs - shift_ci < 264): the contour taps of the 8 harmonics (8 x 39 = 312)
  // cover only 176 distinct bin offsets, the onset clusters of the upper harmonics overlap too.  A tile therefore
  // holds the SUM over the channels: tile for time tap dt, K rows [clip_lo, 16) of the 16 bins that start at bin
  // 8*c, frequency tile ft (rows below clip_lo belong to the previous step when the last chunk pair is clamped).
  auto find_or_add = [&](int dt, int c, int ft, int clip_lo) -> int {
    bool any = false;
    std::fill(scratch.begin(), scratch.end(), (uint16_t)0);
    for (int kk = clip_lo; kk < 16; ++kk) {
      const int u = 8 * c + kk;  // bin of y
      if (u >= sp.data_bins) continue;
      for (int n = 0; n < 128; ++n) {
        const int fl = n / sp.COUT, co = n % sp.COUT;
        const int f = ft * sp.FLT + fl;  // (columns f >= WOUT are computed like the others and dropped by the epilogue)
        double acc = 0.0;
        bool hit = false;
        for (int ci = 0; ci < sp.n_ci; ++ci) {
          const int gg = u - sp.shifts[ci];  // bin of the stacked image
          const int df = gg - sp.SF * f + sp.PL;
          if (df < 0 || df >= sp.KW || gg < 0 || gg >= kContourBins) continue;
          acc += (double)W[((co * sp.n_ci + ci) * sp.KH + dt) * sp.KW + df];
          hit = true;
        }
        if (!hit) continue;
        const float w = (float)acc;
        const uint16_t hi = f2bf(w);
        const uint16_t lo = f2bf(w - bf2f(hi));
        const size_t o = (size_t)(kk >> 3) * 128 * 8 + (size_t)n * 8 + (kk & 7);
        scratch[o] = hi;
        scratch[2048 + o] = lo;
        any = true;
      }
    }
    if (!any) return -1;
    uint64_t h = 1469598103934665603ull;
    for (uint16_t v : scratch) h = (h ^ v) * 1099511628211ull;
    for (int id : by_hash[h])
      if (std::memcmp(tiles.data() + (size_t)id * (kTileBytes / 2), scratch.data(), kTileBytes) == 0) return id;
    tiles.insert(tiles.end(), scratch.begin(), scratch.end());
    by_hash[h].push_back(n_keys);
    return n_keys++;
  };

  // groups: pairs {g, g + G0} (or singles)
  group_step_off.push_back(0);
  n_uses = 0;
  for (int ft_a = 0; ft_a < stride; ++ft_a) {
    const int ft_b = ft_a + stride < n_ft ? ft_a + stride : -1;
    const int fts[2] = {ft_a, ft_b};
    group_ft.push_back(ft_a);
    group_ft.push_back(ft_b);
    struct Use {
      int tile, slot, c8, dt, off;
    };
    std::vector<Use> uses;
    for (int dt = 0; dt < sp.KH; ++dt) {
      std::vector<Use> cand;
      for (int slot = 0; slot < 2; ++slot) {
        const int ft = fts[slot];
        if (ft < 0) continue;
        // 8-bin blocks of y this frequency tile reads through any channel
        std::vector<bool> need(sp.chunks8, false);
        for (int ci = 0; ci < sp.n_ci; ++ci)
          for (int fl = 0; fl < sp.FLT; ++fl) {
            const int f = ft * sp.FLT + fl;
            if (f >= sp.WOUT) continue;
            for (int df = 0; df < sp.KW; ++df) {
              const int gg = sp.SF * f - sp.PL + df, u = gg + sp.shifts[ci];
              if (gg < 0 || gg >= kContourBins || u < 0 || u >= sp.data_bins) continue;
              need[u / 8] = true;
            }
          }
        // cover the needed blocks with K = 16 steps (two adjacent blocks), left to right
        for (int c8 = 0; c8 < sp.chunks8;) {
          if (!need[c8]) {
            ++c8;
            continue;
          }
          const int c = std::min(c8, sp.chunks8 - 3);  // both k-chunks of the step must exist in the data tile, which
                                                       // holds chunks 0 .. chunks8 - 2 (the last one is padding only)
          const int off = 8 * c - sp.SF * sp.FLT * ft;
          const int tile = find_or_add(dt, c, ft, 8 * (c8 - c));
          if (tile >= 0) cand.push_back(Use{tile, slot, c, dt, off});
          c8 += 2;
        }
      }
      std::stable_sort(cand.begin(), cand.end(), [](const Use& a, const Use& b) {
        return a.off != b.off ? a.off < b.off : (a.tile != b.tile ? a.tile < b.tile : a.slot < b.slot);
      });
      uses.insert(uses.end(), cand.begin(), cand.end());
    }
    struct Step {
      int tile;
      uint32_t w[2];
    };
    std::vector<Step> steps;
    size_t i = 0;
    while (i < uses.size()) {
      size_t j = i;
      while (j < uses.size() && uses[j].tile == uses[i].tile && (j == i || uses[j].slot != uses[j - 1].slot)) ++j;
      Step stp{uses[i].tile, {kNoUse, kNoUse}};
      for (size_t u = i; u < j; ++u) {
        stp.w[uses[u].slot] = (uint32_t)(uses[u].c8 * lbo16 + uses[u].dt);  // A start offset >> 4: chunk c8, row dt
        ++n_uses;
      }
      steps.push_back(stp);
      i = j;
    }
    // Software skew between the two slots of a group: the steps only slot 0 uses come first, then the shared ones, then
    // those only slot 1 uses.  Slot 1's next accumulator region is the one slot 0's previous tile still occupies until
    // its conv2 MMAs are done (three regions for four tiles in flight); this way slot 0's tile finishes — and frees its
    // region — early, and slot 1 needs its region late (the issuing warp acquires it at its first use), so neither waits.
    std::stable_sort(steps.begin(), steps.end(), [](const Step& a, const Step& b) {
      auto cls = [](const Step& s) { return s.w[1] == kNoUse ? 0 : (s.w[0] == kNoUse ? 2 : 1); };
      return cls(a) < cls(b);
    });
    bool seen[2] = {false, false};
    for (Step& stp : steps) {
      for (int sl = 0; sl < 2; ++sl)
        if (stp.w[sl] != kNoUse) {
          if (!seen[sl]) stp.w[sl] |= kUseFirstAcc;
          seen[sl] = true;
        }
      tile_seq.push_back(stp.tile);
      slot_words[0].push_back(stp.w[0]);
      slot_words[1].push_back(stp.w[1]);
    }
    group_step_off.push_back((int)tile_seq.size());
  }
  n_tiles = n_keys;
  n_groups = (int)group_ft.size() / 2;
}

// The MMA programs live in constant memory: the issuing warp indexes them with warp-uniform values, so the words,
// the descriptors derived from them and the loop state stay in uniform registers (no per-use R2UR traffic).
// They depend only on the layer geometry (TcConvSpec), not on the weights.
__constant__ uint32_t c_prog[3][2][tc::kMaxSteps];  // [layer][slot][step]
__constant__ int c_tile_seq[3][tc::kMaxSteps];       // [layer][step] -> weight tile id
__constant__ int c_group_step_off[3][tc::kMaxGroups + 1];
__constant__ int c_group_ft[3][2 * tc::kMaxGroups];
// epilogue constants: conv1 bias, conv2 bias
__constant__ float c_bias1[3][32];
__constant__ float c_bias2[3];
// channel 0 of the onset conv2 multiplies the note posteriorgram (models.py:305: concat[note, onset1]): [dt][df]
__constant__ float c_onset_note_w[9];

void tc_upload_epilogue(const float* contour1_b, const float* onset1_b, const float* note1_b, const float* onset2_w,
                        const float* contour2_b, const float* onset2_b, const float* note2_b, cudaStream_t st) {
  float b[3][32] = {};
  for (int i = 0; i < 8; ++i) b[0][i] = contour1_b[i];
  for (int i = 0; i < 32; ++i) b[1][i] = onset1_b[i], b[2][i] = note1_b[i];
  const float b2[3] = {contour2_b[0], onset2_b[0], note2_b[0]};
  cudaMemcpyToSymbolAsync(c_bias1, b, sizeof(b), 0, cudaMemcpyHostToDevice, st);
  cudaMemcpyToSymbolAsync(c_bias2, b2, sizeof(b2), 0, cudaMemcpyHostToDevice, st);
  cudaMemcpyToSymbolAsync(c_onset_note_w, onset2_w, 9 * sizeof(float), 0, cudaMemcpyHostToDevice, st);
  cudaStreamSynchronize(st);
}

// ------------------------------------------------------------------------------------------------
// The fused second convolution as a second tensor-core contraction (A operand in tensor memory).
// After bias + ReLU the epilogue threads write relu(conv1) of their frame back into the accumulator's own 128 columns as
// a bf16 hi/lo split (two elements per column: per 32-column chunk 16 columns hi, 16 columns lo); element k of the row is
// the accumulator column k = fl * COUT + c.  A K = 16 step therefore covers
//   contour: 2 bins x 8 channels        (step ks = bins 2 ks, 2 ks + 1)
//   onset / note: half the channels of one bin   (step ks = bin ks / 2, channels 16 (ks % 2) ..)
// and it contributes to the partial sums P[j][dt] of only a few output offsets j (frequency taps) of the tile:
//   contour: j = bl + 4 - df  in [2 ks, 2 ks + 5]      onset / note: j = fl + 2 - df in [fl, fl + 2]
// With the conv2 accumulator laid out j-major (column j * JS + dt, JS >= KH2) those are a contiguous WINDOW of columns,
// the same for every step up to its start column: every step multiplies by the same small weight tile
//   B2[kk][j' * JS + dt] = w2[c(kk)][dt][df(kk, j')]          (N = 32 columns; onset 16)
// and only the D start column moves (contour 10 ks, note 8 fl, onset 4 fl) — tcgen05.mma takes any EVEN start column.  The
// windows overlap, so all products accumulate into an accumulator the epilogue zeroes after reading it.
// What is left for the CUDA cores is bias / ReLU / split (5 instructions per value) and the time taps (shuffles).
// ------------------------------------------------------------------------------------------------
struct TcB2 {
  int n_tiles, n2, kh2, js, width;  // weight tiles, their N, time taps, columns per output offset j, accumulator columns
};
// (the D start column of an MMA must be even — an odd one raises a misaligned-address fault — hence js = 4 / 8, not 3 / 7)
__host__ __device__ constexpr TcB2 tc_b2_spec(int epi) {  // epi: 0 / 3 contour, 1 onset, 2 note
  return epi == 1 ? TcB2{2, 16, 3, 4, 32} : epi == 2 ? TcB2{2, 32, 7, 8, 64} : TcB2{1, 32, 5, 5, 104};
}

// tiles: [tile][plane hi/lo][k-chunk 2][n N2][8] bf16 (canonical K-major no-swizzle: LBO = N2 * 16 B, SBO = 128 B)
void tc_build_b2(int epi, const float* w2, std::vector<uint16_t>& out) {
  const TcB2 sp = tc_b2_spec(epi);
  const int tile_elems = 2 * 16 * sp.n2;
  out.assign((size_t)sp.n_tiles * tile_elems, 0);
  for (int tl = 0; tl < sp.n_tiles; ++tl)
    for (int kk = 0; kk < 16; ++kk)
      for (int n = 0; n < sp.n2; ++n) {
        const int jp = n / sp.js, dt = n - jp * sp.js;
        float w = 0.f;
        if (dt >= sp.kh2) continue;
        if (epi == 0 || epi == 3) {  // contour conv2 weights [1][8][5][5]; kk = (bin parity) * 8 + channel
          const int b = kk >> 3, c = kk & 7, df = b + 4 - jp;
          if (jp < 6 && df >= 0 && df < 5) w = w2[(c * 5 + dt) * 5 + df];
        } else {
          const int c = 16 * tl + kk, df = 2 - jp;
          if (jp < 3) w = epi == 1 ? w2[(1 + c) * 9 + dt * 3 + df]  // onset conv2 [1][33][3][3], channel 0 = the note input
                                   : w2[c * 21 + dt * 3 + df];      // note conv2 [1][32][7][3]
        }
        const uint16_t hi = f2bf(w), lo = f2bf(w - bf2f(hi));
        const size_t o = (size_t)tl * tile_elems + (size_t)(kk >> 3) * sp.n2 * 8 + (size_t)n * 8 + (kk & 7);
        out[o] = hi;
        out[o + 16 * sp.n2] = lo;
      }
}

int tc_upload_program(int layer, const TcConvPlan& pl, cudaStream_t st) {
  if (layer < 0 || layer > 2 || (int)pl.tile_seq.size() > tc::kMaxSteps - 1 || pl.n_groups > tc::kMaxGroups) return -1;
  for (int sl = 0; sl < 2; ++sl)
    cudaMemcpyToSymbolAsync(c_prog, pl.slot_words[sl].data(), pl.slot_words[sl].size() * 4,
                            ((size_t)layer * 2 + sl) * tc::kMaxSteps * 4, cudaMemcpyHostToDevice, st);
  cudaMemcpyToSymbolAsync(c_tile_seq, pl.tile_seq.data(), pl.tile_seq.size() * 4, (size_t)layer * tc::kMaxSteps * 4,
                          cudaMemcpyHostToDevice, st);
  cudaMemcpyToSymbolAsync(c_group_step_off, pl.group_step_off.data(), pl.group_step_off.size() * 4,
                          (size_t)layer * (tc::kMaxGroups + 1) * 4, cudaMemcpyHostToDevice, st);
  cudaMemcpyToSymbolAsync(c_group_ft, pl.group_ft.data(), pl.group_ft.size() * 4, (size_t)layer * 2 * tc::kMaxGroups * 4,
                          cudaMemcpyHostToDevice, st);
  return cudaStreamSynchronize(st) == cudaSuccess ? 0 : -1;
}

// ------------------------------------------------------------------------------------------------
// fp32 rows -> bf16 hi/lo planes in the k-chunk-major row layout the MMA reads:
//   dst[plane][q8 (chunks8)][row d (rows_total)][8],  d = lead + b*rows_per_window + t, every other row zero.
// lognorm_split_kernel: the log-magnitude of the CQT kernel -> NormalizedLog (reference: layers/signal.py:177-183:
//   (L - min) / (max - min), 0 when max == min) + folded BatchNorm (models.py:188-189) as the split operand of the
//   contour / onset convs (309 bins -> 40 chunks).  (The fp32 copy is only produced on request: launch_lognorm.)
// The contour posteriorgram reaches the note conv in the same layout (264 bins -> 34 chunks), written by the contour
// epilogue itself.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_split8(const float (&v)[8], __nv_bfloat16* dst, size_t off, size_t plane) {
  __align__(16) __nv_bfloat16 hi[8], lo[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    hi[j] = __float2bfloat16_rn(v[j]);
    lo[j] = __float2bfloat16_rn(v[j] - __bfloat162float(hi[j]));
  }
  *reinterpret_cast<uint4*>(dst + off) = *reinterpret_cast<const uint4*>(hi);
  *reinterpret_cast<uint4*>(dst + plane + off) = *reinterpret_cast<const uint4*>(lo);
}

__global__ void lognorm_split_kernel(const float* __restrict__ y, const unsigned int* __restrict__ minmax,
                                     const float* __restrict__ bn, __nv_bfloat16* __restrict__ dst, int n_windows,
                                     int rows_used, int rows_total /* stride */, int chunks8, int rows_per_window, int lead) {
  // one (row, pair of chunks q8, q8 + chunks8 / 2) per thread: the two 32-byte loads are independent (the kernel is bound by
  // load latency, not bandwidth); rows fastest, so the 16-byte stores of a warp are contiguous
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int half = chunks8 / 2;  // chunks8 is even
  const long long total = (long long)rows_used * half;
  if (idx >= total) return;
  const int d = (int)(idx % rows_used);
  const int qa = (int)(idx / rows_used);
  float v[2][8];
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int j = 0; j < 8; ++j) v[h][j] = 0.f;
  const int m = d - lead;
  if (m >= 0) {
    const int b = m / rows_per_window, t = m - b * rows_per_window;
    if (b < n_windows && t < kFrames) {
      const float bn_scale = __ldg(bn), bn_bias = __ldg(bn + 1);
      const float mn = ordered_to_float(minmax[2 * b]);
      const float mx = __fsub_rn(ordered_to_float(minmax[2 * b + 1]), mn);
      const float* p = y + ((size_t)b * kFrames + t) * kCqtBins;
      float raw[2][8];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int bin = (qa + h * half) * 8 + j;
          raw[h][j] = bin < kCqtBins ? __ldg(p + bin) : 0.f;
        }
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if ((qa + h * half) * 8 + j < kCqtBins) {
            const float q = (mx == 0.f) ? 0.f : __fdiv_rn(__fsub_rn(raw[h][j], mn), mx);
            v[h][j] = __fadd_rn(__fmul_rn(q, bn_scale), bn_bias);
          }
    }
  }
  const size_t plane = (size_t)chunks8 * rows_total * 8;
  store_split8(v[0], dst, ((size_t)qa * rows_total + d) * 8, plane);
  store_split8(v[1], dst, ((size_t)(qa + half) * rows_total + d) * 8, plane);
}

// ------------------------------------------------------------------------------------------------
// The tensor-core kernel
// ------------------------------------------------------------------------------------------------
struct TcArgs {
  const __nv_bfloat16* data;    // [2][chunks8][rows_total][8]
  const uint16_t* tiles;        // [n_tiles][8192 B]
  const uint16_t* b2;           // conv2 weight tiles (tc_build_b2), fused layers
  int dbg_skip_loads;           // -DBP_TC_TRACE builds: the producer only pretends to load weight tiles (timing experiment)
  long long* trace;             // -DBP_TC_TRACE builds: [tile][8] clock64 stamps of CTA 0 (see tc_trace)
  TcOut o;                      // where the results go (kernels.cuh)
  int edge_rows;                // row stride of o.edge: [edge slot][side 2][KE][edge_rows]
  int layer;                    // which constant-memory program (0 contour, 1 onset, 2 note)
  int rows_total, n_mtiles, n_windows;
  int n_groups, n_split;        // an item covers groups [s*n_groups/n_split, (s+1)*n_groups/n_split)
  int data_rows, row0;          // tile rows (128 + KH - 1); first data row of M-tile 0
  int ms, h2;                   // M-tile stride (128 - 2*h2) and time halo of the fused conv2
  int chunks8, rows_per_window;
  int cout, flt, wout, n_ft, g0;
};

// Pipeline trace (debug builds with -DBP_TC_TRACE and BP_TC_TRACE=1 in the environment): CTA 0 stamps, per frequency tile n,
// 0 conv1 region acquired, 1 conv1 MMAs issued, 2 epilogue saw the accumulator, 3 split written back, 4 conv2 MMA warp
// released, 5 conv2 MMAs issued, 6 epilogue saw the conv2 sums, 7 tile finished.
#ifdef BP_TC_TRACE
#define TC_TRACE(n, ev)                                                                                       \
  do {                                                                                                        \
    if (a.trace && blockIdx.x == 0 && (n) < 256u && lane == 0) a.trace[(n) * 8u + (ev)] = clock64();            \
  } while (0)
#else
#define TC_TRACE(n, ev) \
  do {                  \
  } while (0)
#endif

__device__ __forceinline__ float sigmoidf_fast(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }

__device__ __forceinline__ void slot_barrier(int slot) {  // the four epilogue warps of one accumulator slot
  asm volatile("bar.sync %0, 128;" ::"r"(1 + slot) : "memory");
}

// Time taps of the fused conv2 across frames.  The thread of tile row r finishes output frame q = r - H of the tile's row
// space: out[q] = sum_dt P_dt[q + dt - H] = sum_a P_{2H-a}[row r - a], a = 0 .. 2H, i.e. every source is `a` lanes BELOW the
// thread.  Sources inside the warp come by shuffle; lanes < a of warps 1..3 take them from the values the previous warp
// published (lanes 32-a .. 31 -> entries a(a-1)/2 + lane - (32-a)) after the slot barrier (time_edges).  A lane adds
// a = 0, 1, .., 2H in this order in both places, so the rounding of a frame does not depend on its row in the tile.
// (The in-warp part is written out in pitch_tile_taps / contour_tile, the cross-warp part is time_edges.)
template <int H, int NJ>
__device__ __forceinline__ void time_edges(float (&S)[NJ], int quad, int lane, const float* xb /* [3][XF] */, int XF) {
  if (quad == 0) return;
#pragma unroll
  for (int a = 1; a <= 2 * H; ++a) {
    if (lane < a) {  // source `a` rows below: lane 32 - a + lane of the previous warp
      const float* e = xb + (quad - 1) * XF + (a * (a - 1) / 2 + lane) * NJ;
#pragma unroll
      for (int j = 0; j < NJ; ++j) S[j] += e[j];
    }
  }
}

// Edge-buffer slot of the tile range that slot `s` of split `q` walks (it starts at tile g0(q) + s * G0): s * n_split + q.
// The range that ENDS below it is slot s of split q - 1, or, for (s, q) = (1, 0), slot 0 of the last split.

// What the epilogue thread of one frame knows about where its results go.  All stores are coalesced: the 32 lanes of a
// warp hold 32 consecutive frames, and every layout below has the frame index fastest.
//   pitch layers (note / onset)  pitch-major planes  [pitch][frame]
//   contour                      chunk-major         [8-bin chunk][frame][8]  (fp32), same shape as the bf16 hi/lo
//                                split layout [plane][chunk][row][8] that the note conv reads
struct RowOut {
  float* raw;    // pitch layers: raw_pm + b*172 + t        ; contour: raw_cm + (b*172 + t)*8            (nullptr: not stored)
  float* unw;    // pitch layers: unw_pm + unwrapped frame  ; contour: unw_cm + unwrapped frame * 8      (nullptr: not stored)
  __nv_bfloat16* chl;  // contour: chl + data row * 8
  float* edge;   // edge buffer column of this frame: edge + R (nullptr: row not complete / not live)
  const float* note_col;  // EPI 1: note_raw_pm + b*172 + t
  int t;         // frame inside the window (of the OUTPUT frame this thread finishes)
  bool ok;       // live output frame whose time taps are complete in this M-tile
  int e_lo, e_hi;  // edge slots of this range's start and of the range above its end (-1: none)
};

// relu(conv1 + bias) of one accumulator row -> bf16 hi/lo split written back IN PLACE: the A operand of the conv2 MMAs
// (TcB2).  Per 32-column chunk q (elements k = 32 q .. 32 q + 31 of the row): columns [32 q, 32 q + 16) hold the hi
// halves, [32 q + 16, 32 q + 32) the lo halves, two elements per column (element 2 c in the low 16 bits).  Rows that are
// not live frames and the bins >= 264 of the last contour tile become zeros.
template <int LAYER>
__device__ __forceinline__ void convert_tile(uint32_t taddr, bool live, int n_valid) {
#pragma unroll 1
  for (int q = 0; q < 4; ++q) {
    uint32_t v[32];
    tmem_ld32_nowait(taddr + q * 32, v);
    tmem_ld_wait();
    const bool ok = live && q * 32 < n_valid;  // n_valid is a multiple of 32 (contour: 64 in the last tile, else 128)
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int c0 = LAYER == 0 ? ((2 * i) & 7) : 2 * i;  // channel of accumulator column 32 q + 2 i
      const float o0 = ok ? fmaxf(__uint_as_float(v[2 * i]) + c_bias1[LAYER][c0], 0.f) : 0.f;
      const float o1 = ok ? fmaxf(__uint_as_float(v[2 * i + 1]) + c_bias1[LAYER][c0 + 1], 0.f) : 0.f;
      const __nv_bfloat162 h = __floats2bfloat162_rn(o0, o1);
      const uint32_t hu = *reinterpret_cast<const uint32_t*>(&h);
      const __nv_bfloat162 l = __floats2bfloat162_rn(o0 - __uint_as_float(hu << 16), o1 - __uint_as_float(hu & 0xffff0000u));
      hi[i] = hu;
      lo[i] = *reinterpret_cast<const uint32_t*>(&l);
    }
    tmem_st16(taddr + q * 32, hi);
    tmem_st16(taddr + q * 32 + 16, lo);
  }
  tmem_st_wait();
}

// Onset / note layers after the conv2 MMAs: the conv2 accumulator holds, for the thread's frame, P[j][dt] (column
// j * JS + dt) = sum over channels and frequency taps for output offset j = 0 .. 5 (bins 4 ft - 1 + j) and time tap dt.
// Reads them, zeroes the accumulator and hands it back, then sums the time taps: S[j] = sum_dt P[j][dt][frame + dt - H],
// sources inside the warp by shuffle, the top lanes published for the next warp (see time_edges).
template <int KH2>
__device__ __forceinline__ void pitch_tile_taps(uint32_t d2, int lane, int quad, float* pub, uint64_t* d2_empty, float (&S)[6]) {
  const int pub_from = quad < 3 ? 32 : 64;  // the last warp of a slot publishes nothing
  constexpr int JS = KH2 == 7 ? 8 : 4;  // columns per output offset (TcB2::js)
  uint32_t d[48];
  tmem_ld32_nowait(d2, reinterpret_cast<uint32_t(&)[32]>(d[0]));
  if constexpr (KH2 == 7) tmem_ld16_nowait(d2 + 32, reinterpret_cast<uint32_t(&)[16]>(d[32]));
  tmem_ld_wait();
  tmem_zero<32>(d2);
  if constexpr (KH2 == 7) {
    tmem_zero<16>(d2 + 32);
    tmem_zero<8>(d2 + 48);
  }
  tmem_st_wait();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(d2_empty);
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    float s = 0.f;
#pragma unroll
    for (int a = 0; a < KH2; ++a) {
      const float p = __uint_as_float(d[j * JS + (KH2 - 1 - a)]);
      if (a == 0) {
        s += p;
      } else {
        const float v = __shfl_up_sync(0xffffffffu, p, a);
        if (lane >= a) s += v;
        if (lane >= pub_from - a) pub[(a * (a - 1) / 2 + lane - (32 - a)) * 6 + j] = p;
      }
    }
    S[j] = s;
  }
}

// Frequency halo + finish for the onset / note layers (FLT = 4, halo 1): S[j] is the time-complete sum for bin 4 ft - 1 + j.
template <int EPI>
__device__ __forceinline__ void finish_pitch_tile(const TcArgs& a, const RowOut& ro, float (&S)[6], float (&carry)[2], int ft,
                                                  bool first, bool last) {
  constexpr int L = EPI == 1 ? 1 : 2;
  const bool lower = ft > 0;
  if (first) {
    if (lower && ro.edge) {
      float* e = ro.edge + (size_t)(ro.e_lo * 2 + 0) * 2 * a.edge_rows;
      e[0] = S[0];
      e[a.edge_rows] = S[1];
    }
  } else {
    S[0] += carry[0];
    S[1] += carry[1];
  }
  const int jlo = first ? (lower ? 2 : 1) : 0;
  const int jhi = (ft == a.n_ft - 1) ? 5 : 4;  // the last tile also finishes its top bin (no tile above)
  if (ro.ok) {
    float nv[3][6];
    if constexpr (EPI == 1) {  // note frames t-1 .. t+1, pitches 4 ft - 2 .. 4 ft + 3 (zero outside the image); lanes run along t
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        const int f = 4 * ft - 2 + c;
        const bool fin = (unsigned)f < (unsigned)kPitches;
        const float* col = ro.note_col + (size_t)f * a.o.raw_rows;
#pragma unroll
        for (int r = 0; r < 3; ++r)
          nv[r][c] = (fin && (unsigned)(ro.t + r - 1) < (unsigned)kFrames) ? __ldg(col + r - 1) : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      if (j < jlo || j >= jhi) continue;
      const int f = 4 * ft - 1 + j;
      float x = S[j] + c_bias2[L];
      if constexpr (EPI == 1) {
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int df = 0; df < 3; ++df)
            if (j + df < 6) x = fmaf(nv[r][j + df], c_onset_note_w[r * 3 + df], x);  // pitch f + df - 1 = 4 ft - 2 + (j + df)
      }
      const float v = sigmoidf_fast(x);
      if (ro.raw) ro.raw[(size_t)f * a.o.raw_rows] = v;
      if (ro.unw) ro.unw[(size_t)f * a.o.frame_stride] = v;
    }
  }
  carry[0] = S[4];
  carry[1] = S[5];
  if (last && ft < a.n_ft - 1 && ro.edge && ro.e_hi >= 0) {
    float* e = ro.edge + (size_t)(ro.e_hi * 2 + 1) * 2 * a.edge_rows;
    e[0] = S[4];
    e[a.edge_rows] = S[5];
  }
}

// One finished 8-bin chunk of the contour posteriorgram for one frame: bf16 hi/lo into the operand layout of the note
// conv, fp32 into the chunk-major posteriorgram.
__device__ __forceinline__ void store_contour_chunk(const TcArgs& a, const RowOut& ro, int chunk, const float (&v)[8]) {
  store_split8(v, ro.chl, (size_t)chunk * a.o.chl_rows * 8, (size_t)a.o.chl_chunks * a.o.chl_rows * 8);
  const float4 x0 = make_float4(v[0], v[1], v[2], v[3]), x1 = make_float4(v[4], v[5], v[6], v[7]);
  if (ro.raw) {
    float4* d = reinterpret_cast<float4*>(ro.raw + (size_t)chunk * a.o.raw_rows * 8);
    d[0] = x0;
    d[1] = x1;
  }
  if (ro.unw) {
    float4* d = reinterpret_cast<float4*>(ro.unw + (size_t)chunk * a.o.frame_stride * 8);
    d[0] = x0;
    d[1] = x1;
  }
}

// Contour layer after the conv2 MMAs (8 -> 1 channels, 5 x 5 taps, models.py:252-259): the conv2 accumulator holds
//   P[j][dt] (column j * 5 + dt) = sum_{c, df} relu(conv1)[c][t][16 ft + j + df - 4] * w2[c][dt][df]     j = 0 .. 19
// for output bins 16 ft - 2 + j of the thread's frame.  Time taps by shuffles (see time_edges), frequency halo by register
// carry, then sigmoid and the stores.
__device__ __forceinline__ void contour_tile(const TcArgs& a, const RowOut& ro, uint32_t d2, uint64_t* d2_empty, int ft,
                                             bool first, bool last, int quad, int lane, int slot, float* xb,
                                             float (&carry)[4], float (&hold)[6]) {
  float S[20];
  float* pub = xb + quad * tc::tc_smem(3).xchg_floats;
  const int pub_from = quad < 3 ? 32 : 64;  // the last warp of a slot publishes nothing
  // one output offset: its five partial sums p[dt] -> time taps (see time_edges for the cross-warp part)
  auto taps = [&](int j, const float (&p)[5]) {
    float s = 0.f;
#pragma unroll
    for (int ta = 0; ta < 5; ++ta) {  // source row `ta` below the thread's: time tap dt = 4 - ta
      const float x = p[4 - ta];
      if (ta == 0) {
        s += x;
      } else {
        const float v = __shfl_up_sync(0xffffffffu, x, ta);
        if (lane >= ta) s += v;
        if (lane >= pub_from - ta) pub[(ta * (ta - 1) / 2 + lane - (32 - ta)) * 20 + j] = x;
      }
    }
    S[j] = s;
  };
  // tensor-memory loads want their column naturally aligned: columns 0 .. 63 first (j = 0 .. 11 and four values of
  // j = 12), then 64 .. 103
  uint32_t keep[4];
  {
    uint32_t d[64];
    tmem_ld32_nowait(d2, reinterpret_cast<uint32_t(&)[32]>(d[0]));
    tmem_ld32_nowait(d2 + 32, reinterpret_cast<uint32_t(&)[32]>(d[32]));
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 12; ++j) {
      float p[5];
#pragma unroll
      for (int dt = 0; dt < 5; ++dt) p[dt] = __uint_as_float(d[j * 5 + dt]);
      taps(j, p);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) keep[k] = d[60 + k];
  }
  {
    uint32_t d[40];
    tmem_ld32_nowait(d2 + 64, reinterpret_cast<uint32_t(&)[32]>(d[0]));
    {
      uint32_t t8[8];
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                   : "=r"(t8[0]), "=r"(t8[1]), "=r"(t8[2]), "=r"(t8[3]), "=r"(t8[4]), "=r"(t8[5]), "=r"(t8[6]), "=r"(t8[7])
                   : "r"(d2 + 96));
#pragma unroll
      for (int k = 0; k < 8; ++k) d[32 + k] = t8[k];
    }
    tmem_ld_wait();
    // everything is in registers: zero the accumulator and hand it back to the conv2 MMA warp
    tmem_zero<32>(d2);
    tmem_zero<32>(d2 + 32);
    tmem_zero<32>(d2 + 64);
    tmem_zero<8>(d2 + 96);
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(d2_empty);
#pragma unroll
    for (int j = 12; j < 20; ++j) {
      float p[5];
#pragma unroll
      for (int dt = 0; dt < 5; ++dt) {
        const int c = j * 5 + dt;  // column 60 .. 99
        p[dt] = __uint_as_float(c < 64 ? keep[c - 60] : d[c - 64]);
      }
      taps(j, p);
    }
  }
  __syncwarp();
  slot_barrier(slot);
  time_edges<2, 20>(S, quad, lane, xb, tc::tc_smem(3).xchg_floats);
  // frequency halo: S[j] <-> bin 16 ft - 2 + j; bins 16 ft - 2 .. 16 ft + 1 also get the top four sums of the tile below.
  // Finished bins leave in aligned 8-bin chunks: chunk 2 ft - 1 = the six bins held back from the previous tile + j = 0, 1;
  // chunk 2 ft = j = 2 .. 9; j = 10 .. 15 are held for the next tile.  Where a range starts / ends, the four partial sums
  // AND the six finished bins next to them go to the edge buffer (10 values per side); edge_fix_kernel assembles the two
  // chunks around the boundary.
  const bool lower = ft > 0;
  if (first) {
    if (lower && ro.edge) {
      float* e = ro.edge + (size_t)(ro.e_lo * 2 + 0) * 10 * a.edge_rows;
#pragma unroll
      for (int k = 0; k < 4; ++k) e[(size_t)k * a.edge_rows] = S[k];
#pragma unroll
      for (int k = 0; k < 6; ++k) e[(size_t)(4 + k) * a.edge_rows] = sigmoidf_fast(S[4 + k] + c_bias2[0]);  // bins 16 ft + 2 .. + 7
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) S[k] += carry[k];
  }
  float fin[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) fin[j] = sigmoidf_fast(S[j] + c_bias2[0]);
  if (ro.ok) {
    if (!first) {  // chunk 2 ft - 1: bins 16 ft - 8 .. 16 ft - 1
      const float v[8] = {hold[0], hold[1], hold[2], hold[3], hold[4], hold[5], fin[0], fin[1]};
      store_contour_chunk(a, ro, 2 * ft - 1, v);
    }
    if (!first || !lower) {  // chunk 2 ft: bins 16 ft .. 16 ft + 7 (at a range start above tile 0 the fix-up writes it)
      const float v[8] = {fin[2], fin[3], fin[4], fin[5], fin[6], fin[7], fin[8], fin[9]};
      store_contour_chunk(a, ro, 2 * ft, v);
    }
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) hold[k] = fin[10 + k];
#pragma unroll
  for (int k = 0; k < 4; ++k) carry[k] = S[16 + k];
  if (last && ft < a.n_ft - 1 && ro.edge && ro.e_hi >= 0) {
    float* e = ro.edge + (size_t)(ro.e_hi * 2 + 1) * 10 * a.edge_rows;
#pragma unroll
    for (int k = 0; k < 4; ++k) e[(size_t)k * a.edge_rows] = S[16 + k];
#pragma unroll
    for (int k = 0; k < 6; ++k) e[(size_t)(4 + k) * a.edge_rows] = fin[10 + k];  // bins 16 ft + 8 .. + 13
  }
}

template <int EPI>
__global__ void __launch_bounds__(tc::kThreads, 1) conv_tc_kernel(const __grid_constant__ TcArgs a) {
  using namespace tc;
  constexpr bool kFused = EPI != 0;
  constexpr int LAYER = EPI == 3 ? 0 : EPI;  // index into the constant banks
  constexpr TcB2 B2 = tc_b2_spec(EPI);
  constexpr int ND2 = 512 - (int)kD2Base >= 2 * B2.width ? 2 : 1;  // conv2 accumulators that fit behind the ring
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr TcSmem SM = tc_smem(EPI);
  constexpr int kStages = SM.stages, kXchgFloats = SM.xchg_floats;
  static_assert(SM.total() <= kMaxSmem && kStages <= kMaxStages, "dynamic shared memory per CTA");
  unsigned char* s_data = smem;                    // [2 planes][chunks][data_rows][16 B]
  unsigned char* s_w = smem + SM.data_bytes;       // [kStages][8192]
  float* s_x = reinterpret_cast<float*>(s_w + kStages * kTileBytes);  // [slot][buf][warp 3][kXchgFloats]
  unsigned char* s_b2 = reinterpret_cast<unsigned char*>(s_x) + SM.xchg_bytes();  // conv2 weight tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_b2 + SM.b2_bytes);
  uint64_t* full_w = bars;             // [kStages]
  uint64_t* empty_w = bars + kStages;  // [kStages]
  uint64_t* data_full = bars + 2 * kStages;
  uint64_t* data_empty = data_full + 1;
  // Parity waits are only safe when whoever waits for phase k + 1 of a barrier has seen phase k complete.  The regions
  // (and a shared conv2 accumulator) alternate between the two slots irregularly (single-tile groups), so the barriers
  // the epilogue warps wait on are per slot: tmem_full[region][slot], d2_full[slot]; each has one committing warp, one
  // set of waiters and at most one phase outstanding.  The others have a single waiting warp that walks the tiles in order.
  uint64_t* tmem_full = data_full + 2;            // [kRegions][2 slots] conv1 accumulator complete
  uint64_t* tmem_empty = tmem_full + 2 * kRegions;  // [kRegions] region may be overwritten by the next conv1 tile
  uint64_t* a2_full = tmem_empty + kRegions;  // [kRegions] relu(conv1) split written back: conv2 MMAs may start
  uint64_t* d2_full = a2_full + kRegions;     // [2 slots] conv2 partial sums of the slot's current tile complete
  uint64_t* d2_empty = d2_full + 2;           // [2 buffers] conv2 accumulator read and zeroed again
  uint64_t* b2_full = d2_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b2_full + 1);

  // Broadcasting the warp index lets the compiler keep the role branches and the producer / MMA loop state in uniform
  // registers (no R2UR before every UTCHMMA: ~40 instead of ~60 instructions per step).
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t lbo = (uint32_t)a.data_rows * 16u;
  const uint32_t plane_bytes = (uint32_t)(a.chunks8 - 1) * lbo;  // the tile holds chunks 0 .. chunks8 - 2

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_w + s, 1);
      mbar_init(empty_w + s, 2);  // one arrival per conv1 MMA warp
    }
    mbar_init(data_full, 1);
    mbar_init(data_empty, 2);
    for (int i = 0; i < kRegions; ++i) {
      mbar_init(tmem_full + 2 * i, 1);
      mbar_init(tmem_full + 2 * i + 1, 1);
      mbar_init(tmem_empty + i, kFused ? 1 : 4);  // fused: the commit behind the conv2 MMAs; else the four epilogue warps
      mbar_init(a2_full + i, 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(d2_full + i, 1);
      mbar_init(d2_empty + i, 4);
    }
    mbar_init(b2_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  if constexpr (kFused) {  // the conv2 accumulators start out zero (the MMAs only ever accumulate into them)
    if (warp < 8 && (warp >> 2) < ND2) {
      const uint32_t d2 = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kD2Base + (uint32_t)(warp >> 2) * B2.width;
#pragma unroll
      for (int c = 0; c + 8 <= B2.width; c += 8) tmem_zero<8>(d2 + c);
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }

  const int n_items = a.n_mtiles * a.n_split;

  if (warp == kProducerWarp) {
    // ------------------------------ producer ------------------------------
    // The whole warp walks the loop with warp-uniform state; the arrive / copy instructions are predicated on the elected
    // lane.  (With `if (lane == 0)` the compiler put an elect loop and three R2UR around every UBLKCP; the weight ring is
    // paced by this loop's latency per step — adding a division to it slowed the contour kernel by 70 %.)
    const uint32_t leader = elect_one() ? 1u : 0u;
    if constexpr (kFused) {
      constexpr uint32_t b2_bytes = (uint32_t)B2.n_tiles * 2u * 16u * B2.n2 * 2u;
      static_assert(b2_bytes <= (uint32_t)SM.b2_bytes, "conv2 weight tiles");
      bulk_g2s_expect_pred(s_b2, a.b2, b2_bytes, b2_full, leader);
    }
    uint32_t stage = 0, ph_w = 0, ph_d = 0;
    const size_t plane_elems = (size_t)a.chunks8 * a.rows_total * 8;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      const int mt = it / a.n_split, sp = it % a.n_split;
      const int g0 = sp * a.n_groups / a.n_split, g1 = (sp + 1) * a.n_groups / a.n_split;
      mbar_wait_wd(data_empty, ph_d ^ 1, 1);
      const size_t row = (size_t)mt * a.ms + a.row0;
      if (leader) {
        mbar_expect_tx(data_full, 2 * plane_bytes);
        // One 1-D bulk copy per plane and chunk: one 4-D tensor-map box measured 1.6 % slower (its innermost dimension is only
        // 16 B, and a chunk of 2 080 B (contour: 130 rows x 16 B) cannot be split into 128-byte-aligned boxes).
        for (int p = 0; p < 2; ++p)
          for (int c = 0; c < a.chunks8 - 1; ++c)
            bulk_g2s(s_data + p * plane_bytes + c * lbo, a.data + p * plane_elems + ((size_t)c * a.rows_total + row) * 8, lbo,
                     data_full);
      }
      __syncwarp();
      ph_d ^= 1;
      const int s0 = c_group_step_off[a.layer][g0], s1 = c_group_step_off[a.layer][g1];
      int tile = c_tile_seq[a.layer][s0];
      for (int s = s0; s < s1; ++s) {
        const int tile_next = c_tile_seq[a.layer][s + 1];  // (one past the end is inside the array)
        mbar_wait_wd(empty_w + stage, ph_w ^ 1, 2);
#ifdef BP_TC_TRACE
        if (a.dbg_skip_loads) {
          if (leader) mbar_arrive(full_w + stage);
        } else
#endif
          bulk_g2s_expect_pred(s_w + stage * kTileBytes, a.tiles + (size_t)tile * (kTileBytes / 2), kTileBytes, full_w + stage,
                               leader);
        if (++stage == kStages) {
          stage = 0;
          ph_w ^= 1;
        }
        tile = tile_next;
      }
    }
  } else if (warp == kMmaWarp0 || warp == kMmaWarp1) {
    // ------------------------------ conv1 MMA issuers: one warp per accumulator slot ---------------------
    constexpr uint32_t idesc = make_idesc(128, 128);
    const int slot = (warp == kMmaWarp0) ? 0 : 1;
    const uint32_t leader = elect_one() ? 1u : 0u;
    uint32_t stage = 0, ph_w = 0, ph_d = 0;
    uint32_t n = 0;  // frequency tiles issued so far by this CTA (both slots, program order) -> region n % 3
    // descriptor words: low = start >> 4 | (LBO >> 4) << 16 ; high = SBO >> 4 | version 1 << 14 (shared by all)
    const uint32_t desc_hi32 = (128u >> 4) | (1u << 14);
    const uint32_t a_hi_base = ((smem_u32(s_data) >> 4) & 0x3fffu) | ((uint32_t)a.data_rows << 16);
    const uint32_t a_lo_base = a_hi_base + (plane_bytes >> 4);
    const uint32_t b_base = ((smem_u32(s_w) >> 4) & 0x3fffu) | ((2048u >> 4) << 16);
    const uint32_t* prog = c_prog[a.layer][slot];
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      const int sp = it % a.n_split;
      const int g0 = sp * a.n_groups / a.n_split, g1 = (sp + 1) * a.n_groups / a.n_split;
      mbar_wait_wd(data_full, ph_d, 3);
      ph_d ^= 1;
      for (int g = g0; g < g1; ++g) {
        const bool two = c_group_ft[a.layer][2 * g + 1] >= 0;
        const bool mine = slot == 0 || two;
        const uint32_t nm = n + (uint32_t)slot, r = nm % kRegions, u = nm / kRegions;
        bool acquired = !mine;  // the region is acquired at this slot's first use of the group (see TcConvPlan::build)
        const int s0 = c_group_step_off[a.layer][g], s1 = c_group_step_off[a.layer][g + 1];
        const uint32_t d = tmem_base + r * 128u;
        uint32_t w = prog[s0];
        for (int s = s0; s < s1; ++s) {
          const uint32_t w_next = prog[s + 1];  // (one word past the end is inside the array)
          mbar_wait_wd(full_w + stage, ph_w, 5);
          if (w != kNoUse) {
            if (!acquired) {
              mbar_wait_wd(tmem_empty + r, (u & 1u) ^ 1u, 4);
              acquired = true;
              TC_TRACE(nm, 0);
            }
            tc_fence_after();
            const uint32_t off = w & 0x3fffu;
            const uint32_t bl = b_base + stage * (kTileBytes >> 4);
            umma_bf16_x3(d, a_hi_base + off, a_lo_base + off, bl, bl + 256u, desc_hi32, idesc,
                         (w & kUseFirstAcc) ? 0u : 1u, leader);
            umma_commit_pred(empty_w + stage, leader);
          } else if (leader) {
            mbar_arrive(empty_w + stage);
          }
          if (++stage == kStages) {
            stage = 0;
            ph_w ^= 1;
          }
          w = w_next;
        }
        if (mine) umma_commit_pred(tmem_full + 2 * r + slot, leader);  // this tile's conv1 accumulator is complete
        if (mine) TC_TRACE(nm, 1);
        n += two ? 2u : 1u;
      }
      umma_commit_pred(data_empty, leader);  // the data tile may be overwritten
    }
  } else if (warp == kMma2Warp) {
    // ------------------------------ conv2 MMA issuer (A operand = the split relu(conv1) in tensor memory) ----------
    if constexpr (kFused) {
      constexpr uint32_t idesc2 = make_idesc(128, B2.n2);
      constexpr uint32_t tile16 = (2u * 16u * B2.n2 * 2u) >> 4;  // bytes >> 4 of one weight tile (hi + lo planes)
      const uint32_t leader = elect_one() ? 1u : 0u;
      const uint32_t desc_hi32 = (128u >> 4) | (1u << 14);
      const uint32_t b2_base = ((smem_u32(s_b2) >> 4) & 0x3fffu) | ((uint32_t)B2.n2 << 16);  // LBO = N2 * 16 bytes
      uint32_t n = 0;
      mbar_wait_wd(b2_full, 0, 6);
      for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        const int sp = it % a.n_split;
        const int g0 = sp * a.n_groups / a.n_split, g1 = (sp + 1) * a.n_groups / a.n_split;
        for (int g = g0; g < g1; ++g) {
          const int n_here = c_group_ft[a.layer][2 * g + 1] >= 0 ? 2 : 1;
          for (int sl = 0; sl < n_here; ++sl, ++n) {
            const uint32_t r = n % kRegions, u = n / kRegions, b = n % ND2, v = n / ND2;
            mbar_wait_wd(a2_full + r, u & 1u, 7);
            mbar_wait_wd(d2_empty + b, (v & 1u) ^ 1u, 8);
            tc_fence_after();
            TC_TRACE(n, 4);
            const uint32_t areg = tmem_base + r * 128u, dacc = tmem_base + kD2Base + b * (uint32_t)B2.width;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
              const uint32_t ah = areg + (uint32_t)((ks >> 1) * 32 + (ks & 1) * 8);
              // window of conv2 accumulator columns this K step contributes to, and its weight tile (TcB2)
              const uint32_t dcol = EPI == 3 ? 10u * ks : (uint32_t)(B2.js * (ks >> 1));
              const uint32_t bt = b2_base + (EPI == 3 ? 0u : (uint32_t)(ks & 1) * tile16);
              umma_ts_bf16_x3(dacc + dcol, ah, ah + 16u, bt, bt + (tile16 >> 1), desc_hi32, idesc2, leader);
            }
            umma_commit_pred(d2_full + sl, leader);    // conv2 partial sums of this tile are complete
            umma_commit_pred(tmem_empty + r, leader);  // and its region may take the next conv1 tile
            TC_TRACE(n, 5);
          }
        }
      }
    }
  } else {
    // ------------------------------ epilogue (warps 0..3 -> slot 0, warps 4..7 -> slot 1) ------------------------------
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int slot = warp >> 2;
    const int row = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    uint32_t n = 0;
    uint32_t full_bits = 0;  // bit r: parity of the next phase of tmem_full[r][slot]
    uint32_t my_tiles = 0;   // tiles of this slot so far: parity of d2_full[slot]
    uint32_t xbuf = 0;  // exchange buffer of this slot, toggled per tile
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      const int mt = it / a.n_split, sp = it % a.n_split;
      const int g0 = sp * a.n_groups / a.n_split, g1 = (sp + 1) * a.n_groups / a.n_split;
      // conv1 row of this thread (it provides relu(conv1) of that frame to the fused conv2) ...
      const int m = mt * a.ms - a.h2 + row;  // row of the (window, frame) space: m = b * rows_per_window + t
      const int b1 = m >= 0 ? m / a.rows_per_window : 0, t1 = m - b1 * a.rows_per_window;
      const bool live = m >= 0 && (b1 < a.n_windows) && (t1 < kFrames);
      // ... and the output frame it finishes: h2 rows earlier (all time taps of the fused conv2 then lie at or below the
      // thread's own row, see time_edges); rows < 2 h2 of the tile are finished by the previous tile
      const int q = m - a.h2;
      const int b = q >= 0 ? q / a.rows_per_window : 0, t = q - b * a.rows_per_window;
      RowOut ro{};
      float carry[4] = {0.f, 0.f, 0.f, 0.f};
      float hold[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if constexpr (kFused) {
        ro.e_lo = slot * a.n_split + sp;
        ro.e_hi = (sp + 1 < a.n_split) ? slot * a.n_split + sp + 1 : (slot == 0 ? a.n_split : -1);
        ro.ok = row >= 2 * a.h2 && q >= 0 && b < a.n_windows && t < kFrames;
        ro.t = t;
        if (ro.ok) {
          ro.edge = a.o.edge + q;
          int uf = -1;  // unwrapped frame (reference: inference.py:247-279), if this frame is kept
          if (a.o.ud) {
            const UnwrapDesc u = a.o.ud[b];
            const int tt = t - kOverlapHalf;
            if ((unsigned)tt < (unsigned)max(u.rows, 0)) uf = (int)(u.dst_base + tt);
          }
          if constexpr (EPI == 3) {
            ro.chl = a.o.chl + ((size_t)a.o.chl_lead + (size_t)b * a.o.chl_rpw + t) * 8;
            if (a.o.raw) ro.raw = a.o.raw + ((size_t)b * kFrames + t) * 8;
            if (uf >= 0) ro.unw = a.o.unwrapped + (size_t)uf * 8;
          } else {
            if (a.o.raw) ro.raw = a.o.raw + (size_t)b * kFrames + t;
            if (uf >= 0) ro.unw = a.o.unwrapped + uf;
            if constexpr (EPI == 1) ro.note_col = a.o.note_raw + (size_t)b * kFrames + t;
          }
        }
      }
      for (int g = g0; g < g1; ++g) {
        const bool two = c_group_ft[a.layer][2 * g + 1] >= 0;
        const int ft = c_group_ft[a.layer][2 * g + slot];
        const uint32_t nm = n + (uint32_t)slot;
        n += two ? 2u : 1u;
        if (ft < 0) continue;
        const uint32_t r = nm % kRegions;
        mbar_wait_wd(tmem_full + 2 * r + slot, (full_bits >> r) & 1u, 9);
        full_bits ^= 1u << r;
        tc_fence_after();
        if (quad == 0) TC_TRACE(nm, 2);
        const uint32_t taddr = lane_base + r * 128u;
        // first / last tile of this slot's ascending range inside the item
        const bool first = (g == g0);
        const bool last = (g == g1 - 1) || (ft == a.n_ft - 1);
        if constexpr (EPI == 0) {
          // contour: 16 bins x 8 channels, bias + ReLU, channels-last rows of 128 contiguous floats
          const int n_valid = min(a.flt, a.wout - ft * a.flt) * a.cout;
          float* dst = a.o.act + ((size_t)b * kFrames + t) * ((size_t)a.wout * a.cout) + (size_t)ft * 128;
#pragma unroll 1
          for (int c4 = 0; c4 < 4; ++c4) {
            uint32_t v[32];
            tmem_ld32_nowait(taddr + c4 * 32, v);
            tmem_ld_wait();
            if (live) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float4 o;
                o.x = fmaxf(__uint_as_float(v[4 * i + 0]) + c_bias1[0][(4 * i + 0) & 7], 0.f);
                o.y = fmaxf(__uint_as_float(v[4 * i + 1]) + c_bias1[0][(4 * i + 1) & 7], 0.f);
                o.z = fmaxf(__uint_as_float(v[4 * i + 2]) + c_bias1[0][(4 * i + 2) & 7], 0.f);
                o.w = fmaxf(__uint_as_float(v[4 * i + 3]) + c_bias1[0][(4 * i + 3) & 7], 0.f);
                if (c4 * 32 + 4 * i < n_valid) reinterpret_cast<float4*>(dst + c4 * 32)[i] = o;
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tmem_empty + r);
        } else {
          // bias + ReLU + split in place, then the conv2 MMAs take over (kMma2Warp) ...
          const int n_valid = min(a.flt, a.wout - ft * a.flt) * a.cout;
          convert_tile<LAYER>(taddr, live, n_valid);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(a2_full + r);
          if (quad == 0) TC_TRACE(nm, 3);
          // ... and hand back P[j][dt] in the conv2 accumulator
          const uint32_t bb = nm % ND2;
          mbar_wait_wd(d2_full + slot, my_tiles & 1u, 10);
          ++my_tiles;
          tc_fence_after();
          if (quad == 0) TC_TRACE(nm, 6);
          const uint32_t d2 = lane_base + kD2Base + bb * (uint32_t)B2.width;
          float* xb = s_x + (slot * 2 + xbuf) * 3 * kXchgFloats;
          xbuf ^= 1u;
          if constexpr (EPI == 3) {
            contour_tile(a, ro, d2, d2_empty + bb, ft, first, last, quad, lane, slot, xb, carry, hold);
          } else {
            constexpr int KH2 = (EPI == 1) ? 3 : 7, H = KH2 / 2;
            float S[6];
            pitch_tile_taps<KH2>(d2, lane, quad, xb + quad * kXchgFloats, d2_empty + bb, S);
            __syncwarp();
            slot_barrier(slot);
            time_edges<H, 6>(S, quad, lane, xb, kXchgFloats);
            float c2[2] = {carry[0], carry[1]};
            finish_pitch_tile<EPI>(a, ro, S, c2, ft, first, last);
            carry[0] = c2[0];
            carry[1] = c2[1];
          }
          if (quad == 0) TC_TRACE(nm, 7);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// ------------------------------------------------------------------------------------------------
// Where two tile ranges meet (frequency tile ft_b = first tile of a range, ft_b > 0) the 2 * HALO bins
// FLT * ft_b - HALO + k got one partial sum from each side: finish them here.  Pitch layers: 2 bins per frame.  Contour:
// 4 bins, and with the six finished bins each side left next to them the two 8-bin chunks around the boundary.
// ------------------------------------------------------------------------------------------------
struct EdgeFixArgs {
  TcOut o;
  int edge_rows, n_rows;        // rows of the (window, frame) space covered by the M-tiles
  int n_edges;                  // 2 * n_split slots: slot e = s * n_split + q starts at tile q * n_groups / n_split + s * G0
  int n_split, n_groups, g0, n_ft;
  int layer, wout, rows_per_window, n_windows;
};

__global__ void edge_fix_kernel(const EdgeFixArgs a) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_edge = a.layer == 0 ? 1 : 2;  // contour: one thread per (frame, edge); pitch layers: per (frame, edge, bin)
  const long long total = (long long)a.n_rows * a.n_edges * per_edge;
  if (idx >= total) return;
  const int R = (int)(idx % a.n_rows);  // rows fastest: coalesced reads of the edge buffer, coalesced stores
  const int ek = (int)(idx / a.n_rows);
  const int e = ek / per_edge, k = ek - e * per_edge;
  const int b = R / a.rows_per_window, t = R - b * a.rows_per_window;
  if (b >= a.n_windows || t >= kFrames) return;
  const int es = e / a.n_split, eq = e - es * a.n_split;
  const int ft_b = eq * a.n_groups / a.n_split + es * a.g0;
  if (ft_b <= 0 || ft_b >= a.n_ft) return;  // not a boundary between two ranges
  int uf = -1;
  if (a.o.ud) {
    const UnwrapDesc u = a.o.ud[b];
    const int tt = t - kOverlapHalf;
    if ((unsigned)tt < (unsigned)max(u.rows, 0)) uf = (int)(u.dst_base + tt);
  }
  if (a.layer == 0) {
    const float* lo = a.o.edge + (size_t)(e * 2 + 0) * 10 * a.edge_rows + R;  // from the range that starts at ft_b
    const float* hi = a.o.edge + (size_t)(e * 2 + 1) * 10 * a.edge_rows + R;  // from the range that ends at ft_b - 1
    float fx[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)  // (S + carry) + bias, the order of the in-kernel carry
      fx[q] = sigmoidf_fast((lo[(size_t)q * a.edge_rows] + hi[(size_t)q * a.edge_rows]) + c_bias2[0]);
    float va[8], vb[8];
#pragma unroll
    for (int q = 0; q < 6; ++q) {
      va[q] = hi[(size_t)(4 + q) * a.edge_rows];      // bins 16 ft_b - 8 .. - 3
      vb[2 + q] = lo[(size_t)(4 + q) * a.edge_rows];  // bins 16 ft_b + 2 .. + 7
    }
    va[6] = fx[0], va[7] = fx[1], vb[0] = fx[2], vb[1] = fx[3];
    __nv_bfloat16* chl = a.o.chl + ((size_t)a.o.chl_lead + (size_t)b * a.o.chl_rpw + t) * 8;
    const size_t plane = (size_t)a.o.chl_chunks * a.o.chl_rows * 8;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int chunk = 2 * ft_b - 1 + c;
      const float(&v)[8] = c ? vb : va;
      store_split8(v, chl, (size_t)chunk * a.o.chl_rows * 8, plane);
      const float4 x0 = make_float4(v[0], v[1], v[2], v[3]), x1 = make_float4(v[4], v[5], v[6], v[7]);
      if (a.o.raw) {
        float4* d = reinterpret_cast<float4*>(a.o.raw + ((size_t)chunk * a.o.raw_rows + (size_t)b * kFrames + t) * 8);
        d[0] = x0, d[1] = x1;
      }
      if (uf >= 0) {
        float4* d = reinterpret_cast<float4*>(a.o.unwrapped + ((size_t)chunk * a.o.frame_stride + uf) * 8);
        d[0] = x0, d[1] = x1;
      }
    }
    return;
  }
  const int f = 4 * ft_b - 1 + k;
  if (f < 0 || f >= a.wout) return;
  float x = (a.o.edge[((size_t)(e * 2 + 0) * 2 + k) * a.edge_rows + R] +
             a.o.edge[((size_t)(e * 2 + 1) * 2 + k) * a.edge_rows + R]) + c_bias2[a.layer];  // (S + carry) + bias
  if (a.o.note_raw) {
#pragma unroll
    for (int dt = 0; dt < 3; ++dt)
#pragma unroll
      for (int df = 0; df < 3; ++df) {
        const int tt = t + dt - 1, ff = f + df - 1;
        if ((unsigned)tt < (unsigned)kFrames && (unsigned)ff < (unsigned)kPitches)
          x = fmaf(__ldg(a.o.note_raw + (size_t)ff * a.o.raw_rows + (size_t)b * kFrames + tt), c_onset_note_w[dt * 3 + df], x);
      }
  }
  const float v = sigmoidf_fast(x);
  if (a.o.raw) a.o.raw[(size_t)f * a.o.raw_rows + (size_t)b * kFrames + t] = v;
  if (uf >= 0) a.o.unwrapped[(size_t)f * a.o.frame_stride + uf] = v;
}

// ------------------------------------------------------------------------------------------------
int tc_rows_total(int n_windows, int rows_per_window) {
  // lead rows + the rows of the windows + what the last (overlapping) M-tile and its time taps may touch
  return n_windows * rows_per_window + tc::kMTile + 16;
}

int tc_setup() {
  cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::tc_smem(0).total());
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::tc_smem(1).total());
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::tc_smem(2).total());
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::tc_smem(3).total());
  return e == cudaSuccess ? 0 : -1;
}

void launch_lognorm_split(const float* y, const unsigned int* minmax, const float* bn, __nv_bfloat16* dst,
                          const TcConvSpec& sp, int n_windows, int rows_stride, cudaStream_t st) {
  const int rows_used = tc_rows_total(n_windows, sp.rows_per_window);  // <= rows_stride
  const long long cells = (long long)rows_used * (sp.chunks8 / 2);  // a thread converts two chunks of a row
  lognorm_split_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(y, minmax, bn, dst, n_windows, rows_used, rows_stride,
                                                                       sp.chunks8, sp.rows_per_window, sp.lead_rows);
}

size_t tc_edge_floats(const TcConvSpec& sp, int n_windows) {
  const int ms = tc::kMTile - (sp.KH2 - 1);
  const int n_mtiles = (n_windows * sp.rows_per_window + ms - 1) / ms;
  const int per_side = sp.epi == 0 ? 10 : 2;
  return (size_t)2 * sp.G0 * 2 * per_side * ((size_t)n_mtiles * ms);  // at most 2 * G0 range starts
}

void launch_conv_tc(const __nv_bfloat16* data, const TcConvDev& dev, const TcOut& o, int n_windows, int rows_stride,
                    int n_sms, cudaStream_t st, bool fuse_next) {
  const TcConvSpec& sp = dev.spec;
  const bool fused = sp.epi != 0 || fuse_next;
  TcArgs a{};
  a.data = data;
  a.tiles = dev.tiles;
  a.b2 = dev.b2;
  a.o = o;
  a.layer = dev.layer;
  a.rows_total = rows_stride;  // row stride of the split layout (fixed per model, independent of the batch)
  a.h2 = fused ? (sp.KH2 - 1) / 2 : 0;
  a.ms = tc::kMTile - 2 * a.h2;
  a.n_mtiles = (n_windows * sp.rows_per_window + a.ms - 1) / a.ms;
  a.edge_rows = a.n_mtiles * a.ms;
  a.n_windows = n_windows;
  a.n_groups = dev.n_groups;
  // An item is (M-tile, one of `split` runs of frequency groups).  Pick the split that minimises the number of waves
  // times the work per item, the data-tile load counted as half a group: full chunks run unsplit, partial chunks and
  // small batches spread over all SMs.
  int split = 1;
  double best = 1e30;
  for (int s = 1; s <= dev.n_groups; ++s) {
    const int waves = (a.n_mtiles * s + n_sms - 1) / n_sms;
    const double cost = waves * ((dev.n_groups + s - 1) / s + 0.5);
    if (cost < best - 1e-9) best = cost, split = s;
  }
  a.n_split = split;
  a.data_rows = tc::kMTile + sp.KH - 1;
  a.row0 = sp.lead_rows - sp.PT - a.h2;
  a.chunks8 = sp.chunks8;
  a.rows_per_window = sp.rows_per_window;
  a.cout = sp.COUT;
  a.flt = sp.FLT;
  a.wout = sp.WOUT;
  a.n_ft = (sp.WOUT + sp.FLT - 1) / sp.FLT;
  a.g0 = sp.G0;
  const int n_items = a.n_mtiles * a.n_split;
  const int grid = n_items < n_sms ? n_items : n_sms;
#ifdef BP_TC_TRACE
  static long long* d_trace = nullptr;
  const bool tracing = getenv("BP_TC_TRACE") != nullptr;
  if (tracing) {
    if (!d_trace) cudaMalloc(&d_trace, 256 * 8 * sizeof(long long));
    cudaMemsetAsync(d_trace, 0, 256 * 8 * sizeof(long long), st);
    a.trace = d_trace;
  }
  a.dbg_skip_loads = getenv("BP_TC_SKIP_LOADS") != nullptr;
#endif
  if (sp.epi == 0 && fuse_next)
    conv_tc_kernel<3><<<grid, tc::kThreads, tc::tc_smem(3).total(), st>>>(a);
  else if (sp.epi == 0)
    conv_tc_kernel<0><<<grid, tc::kThreads, tc::tc_smem(0).total(), st>>>(a);
  else if (sp.epi == 1)
    conv_tc_kernel<1><<<grid, tc::kThreads, tc::tc_smem(1).total(), st>>>(a);
  else
    conv_tc_kernel<2><<<grid, tc::kThreads, tc::tc_smem(2).total(), st>>>(a);
#ifdef BP_TC_TRACE
  if (tracing) {
    static long long h[256 * 8];
    cudaMemcpyAsync(h, d_trace, sizeof(h), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    long long t0 = h[0];
    fprintf(stderr, "tc_trace layer %d n_items %d split %d grid %d\n", dev.layer, n_items, a.n_split, grid);
    for (int n = 0; n < 256 && h[n * 8 + 1]; ++n) {
      fprintf(stderr, "tile %3d:", n);
      for (int e = 0; e < 8; ++e) fprintf(stderr, " %8lld", h[n * 8 + e] ? h[n * 8 + e] - t0 : -1);
      fprintf(stderr, "\n");
    }
  }
#endif
  if (fused) {  // slot s of split q covers tiles [g0(q) + s*G0, g1(q) + s*G0): edge slot s*split + q
    EdgeFixArgs ef{};
    ef.o = o;
    ef.edge_rows = a.edge_rows;
    ef.n_rows = n_windows * sp.rows_per_window;
    ef.n_edges = 2 * split;
    ef.n_split = split;
    ef.n_groups = dev.n_groups;
    ef.g0 = sp.G0;
    ef.n_ft = a.n_ft;
    ef.layer = sp.epi;  // c_bias2 index: 0 contour, 1 onset, 2 note
    ef.wout = sp.WOUT;
    ef.rows_per_window = sp.rows_per_window;
    ef.n_windows = n_windows;
    const long long total = (long long)ef.n_rows * ef.n_edges * (sp.epi == 0 ? 1 : 2);
    edge_fix_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ef);
  }
}

}  // namespace bp
