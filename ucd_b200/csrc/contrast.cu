// Fused PixelConLossV2 (utils/loss.py:412-466) with the joint-probability weights of
// pre_contrastive_pixel (utils/loss.py:369-393) computed in-kernel.  The N_a x N_c similarity,
// mask and P matrices are never materialised.
//
// Math (SURVEY.md Appendix A.2).  For anchor row i and contrast column j:
//   s_ij = a_i.c_j / tau ; same_ij = [la_i == lc_j] ; mp_ij = same_ij - [j is i itself]
//   neg_i = sum_j (1-same_ij) exp(s_ij)   (unshifted) ;  m_i = max_j s_ij ;  num_i = sum_j mp_ij
//   den_ij = exp(s_ij - m_i) + neg_i ;  w_ij = mp_ij * P_ij
//   L_i = sum_j w_ij (s_ij - m_i - log den_ij) ;  loss = mean_{num_i != 0} ( -L_i / num_i )
//   d(-L_i/num_i)/d a_i = (T_i V_i - U_i) / (tau num_i)
//      V_i = sum_j (1-same_ij) exp(s_ij) c_j ;  T_i = sum_j w_ij / den_ij ;  U_i = sum_j w_ij neg_i/den_ij c_j
//
// Two tensor-core sweeps over the column tiles, same kernel template:
//   sweep 1: S = A C^T (tcgen05, K=256) -> epilogue: exp, masks, row max/neg/num; E = masked exp(S)
//            in bf16 -> a separate E region of tensor memory -> V += E C (tcgen05 TS with the SAME C tile read MN-major).
//   sweep 2: S again and P = pA pC^T (K = padded C_old) -> epilogue: den, log, weights, L_i, T_i;
//            Ucoef in bf16 -> the consumed P columns -> U += Ucoef C.
// The gradient needs no third sweep: backward is a scaled copy of (T V - U)/(tau num).
//
// CTA = one 128-row block x one contiguous range of column tiles ("split").  Warp roles: warp 0 issues
// bulk async copies (TMA engine) of pre-tiled bf16 operands, warp 1 owns TMEM and issues the S (and P) MMAs,
// warp 2 issues the V / U MMAs (A operand = E / Ucoef read from tensor memory), warps 3-10 are the epilogue
// (two per SM sub-partition; one thread per row and column half, accumulators read with tcgen05.ld, E / Ucoef
// written back with tcgen05.st).  The issuing warps run warp-uniform with the instructions in elect_one_sync() blocks
// (umma.cuh).  Everything is handed over through mbarriers; no __syncthreads in the tile loop.
// Column tiles stream through a ring of half-tile slots (below); S is a single accumulator that is released as soon
// as the epilogue holds it in registers.
//
// Why not cta_group::2 (M = 256 over a CTA pair sharing the column tile)?  One tcgen05.mma.cta_group::2 carries ONE
// B descriptor that both CTAs apply to their own shared memory, each supplying HALF of B's N extent.  For S = A C^T the
// N extent is the tile's 128 COLUMNS (CTA r would hold columns 64r..64r+63, all 256 features); for V = E C the N extent
// is the 256 FEATURES (CTA r would hold features 128r..128r+127 of all 128 columns).  Per CTA that is three of the four
// 16 KB (column half x feature half) quadrants, and because both CTAs must find their S half and their V half at the
// same offsets, the quadrant they have in common (own columns x own features) cannot serve both views in both CTAs at
// once: four 16 KB regions with one duplicate = the same 64 KB per tile as now.  Rotating the rows of CTA 1's copy
// fixes the S view but then position p of V's K axis means column p in CTA 0 and column p+64 in CTA 1.  And all
// tcgen05 instructions of a kernel must use the same cta_group, so S cannot be paired while V stays per CTA.  With
// the same 24 MMAs per 2048 clk of pipe work the pair would not relieve the issue side either.
#include "umma.cuh"
#ifdef UCD_DEBUG_KNOBS
#include "../../include/ucd_b200_debug.h"
#endif

#include <stdlib.h>

namespace ucd {

constexpr int kEpiWarps = 8;                       // 2 per SM sub-partition: one hides the other's stalls
constexpr int kConThreads = 96 + 32 * kEpiWarps;   // producer warp + two MMA-issuing warps + epilogue warps
constexpr uint32_t kTileBytes = 65536;  // 128 rows x 256 bf16
constexpr uint32_t kChunkB = 2048;      // one 8-element k-chunk for 128 rows
constexpr uint32_t kESub = 16384;       // 128 rows x 64 columns bf16

constexpr uint32_t kSlotBytes = 32768;  // half a column tile: 16 of its 32 k-chunks (128 features) x 128 columns

// shared memory map (bytes)
constexpr uint32_t OFF_A = 0;
constexpr uint32_t OFF_C = 65536;     // ring of half-tile slots: 5 in sweep 1, 4 in sweep 2 (the 5th is OFF_E there)
constexpr uint32_t OFF_E = 196608;    // 32 KB: sweep 2 probability operands
constexpr uint32_t OFF_PA = OFF_E;    // sweep 2: row probabilities [kpad/8][128][8] bf16 (kpad*256 B <= 28 KB)
constexpr uint32_t kProbBytes = 32768;  // OFF_PA .. OFF_LAB: the column probabilities use what pA leaves, in K chunks
constexpr uint32_t OFF_LAB = 229376;  // 3 x 128 int32 (labels of the up to three column tiles in flight)
constexpr uint32_t OFF_BAR = 230912;
constexpr uint32_t kConSmem = OFF_BAR + 256;
constexpr int kMaxChunks = 16;        // ranks whose columns are gathered (one 8-GPU box: 8)
constexpr int kMaxTilesPerCta = 4096;  // column tiles one CTA walks (bit mask in shared memory)

// Column tiles stream through a RING of half-tile slots (feature halves: k-chunks 0-15 / 16-31 of the tile, 32 KB each).
// A tile's two slots stay occupied from their load until the V/U MMAs of the tile have retired (V reads every feature
// of 16 columns per K step), i.e. for load + S + epilogue + V; with whole-tile stages only two fit beside the 64 KB
// anchor tile and every second tile waited ~750 clk for its stage (profiles/r02a_*).  Five half slots keep 2.5 tiles
// in flight: the first half of tile t+2 is loaded - and its 8 S K-steps issued - while tile t still holds its slots.
//
// A: row tile loaded | HF[2*slot+q]: 16 KB quarter q (4 K steps of S) of a slot has landed | HE[slot]: slot empty
// (tcgen05.commit of the tile's last V/U MMA + the 8 epilogue warps, which read the tile's labels) | SF: S accumulator
// ready | SE: S buffer free | EF[(buf*2+half)*2+chunk]: 32 columns of E/Ucoef written to TMEM (2 K steps of V/U) |
// PF/PE: probability stage full/empty | V: all MMAs retired | SR (sweep 2): S accumulator is in the epilogue's registers
enum { BAR_A = 0, BAR_HF = 1, BAR_HE = 11, BAR_SF = 16, BAR_SE = 18, BAR_EF = 20, BAR_PF = 28, BAR_PE = 29, BAR_V = 30,
       BAR_SR = 31 };

// position in the slot ring: slot index and the parity of its use count
template <int NSLOT>
struct Ring {
  int slot = 0;
  uint32_t par = 0;
  __device__ __forceinline__ void next() {
    if (++slot == NSLOT) {
      slot = 0;
      par ^= 1u;
    }
  }
};

struct ConArgs {
  const __nv_bfloat16* feat_tiles;
  const __nv_bfloat16* prob_tiles;
  const int* lab_tiles;
  const int* chunk_counts;  // chunk c: {N_a, N_o} at chunk_counts + c * (chunk_stride ? chunk_stride / 4 : 2)
  int n_chunks;
  long long chunk_tiles;
  // chunk_stride > 0: the five column arrays of chunk c (one rank's exchange payload) start chunk_stride bytes after
  // those of chunk c-1 (pointers address chunk `chunk_origin`); 0: every array is [n_chunks][chunk_tiles][...] on its own
  long long chunk_stride;
  int chunk_origin;
  int chunk_lo, chunk_hi, chunk_skip;  // this launch walks the columns of chunks [lo, hi) except `skip`
  int split_base;                      // first partial slot of this launch (sweep 1 may run as two launches)
  const __nv_bfloat16* row_feat;  // row (anchor) tiles: [row_block][32][128][8]
  const __nv_bfloat16* row_prob;  // [row_block][kpad/8][128][8]
  const int* row_lab;             // [row_block][128]
  const int* n_rows;              // device scalar: number of valid rows
  const int* tile_range;          // [tiles][2] min/max valid label of every column tile (sweep 2 skip test)
  const int* row_range;           // [row_block][2] same for the row tiles
  long long self_tile0;           // column tile holding row block 0 itself (block rb <-> self_tile0 + rb), -1: none
  const int* min_new;
  const float* dense_p;
  long long ldp;
  float inv_tau;
  int splits;
  int need_grad;
  int kpad;
  long long rows_pad;
  float* stats_part;   // [splits][3][rows_pad]   sweep 1 out: raw row max, neg, num
  float* acc_part;     // [splits][rows_pad][256] sweep 1: V ; sweep 2: U
  const float* stats;  // [3][rows_pad]           sweep 2 in (combined)
  float* loss_part;    // [splits][2][rows_pad]   sweep 2 out: L_i, T_i
  long long* trace;    // debug: [grid][16] cycle counters per role (ucd_con_debug_trace), or NULL
  // self-contrast losses (PixelConLoss v1 / SupConLoss, utils/loss_new.py:263-400; see sweep3_cols)
  int shift;           // sweep 2: 1 = PixelConLossV2's exp(s - m) in the denominator, 0 = unshifted (v1)
  const float* col_a;  // sweep 3: per-pixel coefficients in column (= row) order, see sweep3_cols
  const float* col_b;
  const float* col_c;
};

// mbar_wait that also accumulates the cycles spent waiting (debug tracing of the role pipelines)
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, long long& acc) {
  const long long c0 = clock64();
  mbar_wait(bar, parity);
  acc += clock64() - c0;
}

struct TileLoc {
  long long gtile;  // tile index in global numbering: chunk * chunk_tiles + tile within the chunk
  int nvalid;       // valid columns in this tile (1..128)
  long long dcol0;  // first column in "dense" numbering (single-chunk compat path)
  int c, lt;        // chunk and tile within the chunk
};

// byte offset of tile (c, lt) of a column array with `tile_bytes` per tile
__device__ __forceinline__ size_t tile_off(const TileLoc& t, size_t tile_bytes, long long chunk_tiles, long long chunk_stride,
                                           int chunk_origin) {
  return chunk_stride ? (size_t)((long long)(t.c - chunk_origin) * chunk_stride) + (size_t)t.lt * tile_bytes
                      : (size_t)((long long)(t.c - chunk_origin) * chunk_tiles + t.lt) * tile_bytes;
}

__device__ __forceinline__ TileLoc locate_tile(int k, const int* pre, const int* ncols, int n_chunks,
                                               long long chunk_tiles) {
  int c = 0;
  while (c + 1 < n_chunks && k >= pre[c + 1]) ++c;
  const int lt = k - pre[c];
  TileLoc t;
  t.gtile = (long long)c * chunk_tiles + lt;
  t.nvalid = min(128, ncols[c] - lt * 128);
  t.dcol0 = (long long)lt * 128;
  t.c = c, t.lt = lt;
  return t;
}

// The tile loops visit their tiles in increasing order: the chunk a tile belongs to is tracked in registers and only
// advanced (shared-memory reads) when a chunk boundary is crossed.  (locate_tile per tile - a dependent chain of
// shared-memory loads and branches - cost every epilogue warp ~300 clk per tile, ncu source view r02.)
struct TileCursor {
  int c, base, next, ncols;
  long long chunk_tiles;
  const int* pre;
  const int* ncols_arr;
  int n_chunks;
  __device__ __forceinline__ void init(const int* pre_, const int* ncols_, int n_chunks_, long long chunk_tiles_) {
    pre = pre_, ncols_arr = ncols_, n_chunks = n_chunks_, chunk_tiles = chunk_tiles_;
    c = 0, base = 0, next = pre_[1], ncols = ncols_[0];
  }
  __device__ __forceinline__ TileLoc seek(int k) {  // k must not decrease between calls
    while (c + 1 < n_chunks && k >= next) {
      ++c;
      base = next;
      next = pre[c + 1];
      ncols = ncols_arr[c];
    }
    const int lt = k - base;
    TileLoc t;
    t.gtile = (long long)c * chunk_tiles + lt;
    t.nvalid = min(128, ncols - lt * 128);
    t.dcol0 = (long long)lt * 128;
    t.c = c, t.lt = lt;
    return t;
  }
};

__device__ __forceinline__ uint32_t bf16x2_bits(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// ---- sweep 1 epilogue on 32 columns ---------------------------------------------------------
template <bool FULL, bool SELF>
__device__ __forceinline__ void sweep1_cols(const uint32_t (&r)[32], const int* __restrict__ lab, int cbase, int nv,
                                            int la, int rself, float sc, float& mx, float& neg, float& num,
                                            uint32_t (&pk)[16]) {
#pragma unroll
  for (int j4 = 0; j4 < 32; j4 += 4) {
    const int4 l4 = *reinterpret_cast<const int4*>(lab + cbase + j4);
    const int ls[4] = {l4.x, l4.y, l4.z, l4.w};
    float e[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int col = cbase + j4 + u;
      const float acc = __uint_as_float(r[j4 + u]);
      const bool same = ls[u] == la;
      float ev = same ? 0.f : ex2f(acc * sc);
      float cnt = same ? 1.f : 0.f;
      float mv = acc;
      if (!FULL) {
        const bool ok = col < nv;
        ev = ok ? ev : 0.f;
        cnt = ok ? cnt : 0.f;
        mv = ok ? acc : -3.0e38f;
      }
      if (SELF) cnt -= (col == rself) ? 1.f : 0.f;
      mx = fmaxf(mx, mv);
      neg += ev;
      num += cnt;
      e[u] = ev;
    }
    pk[j4 / 2] = bf16x2_bits(e[0], e[1]);
    pk[j4 / 2 + 1] = bf16x2_bits(e[2], e[3]);
  }
}

// Sweep-1 fast path: the tile's label range misses the row block's, so every pair is a negative - no label
// compare, no positive count: exp, row sum, row max, pack (about 4.5 instructions per pair).
__device__ __forceinline__ void sweep1_cols_neg(const uint32_t (&r)[32], float sc, float& mx, float& neg,
                                                uint32_t (&pk)[16]) {
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    const float a0 = __uint_as_float(r[j]), a1 = __uint_as_float(r[j + 1]);
    const float e0 = ex2f(a0 * sc), e1 = ex2f(a1 * sc);  // (a polynomial exp2 on the FMA pipe for half of them was slower)
    mx = fmaxf(mx, fmaxf(a0, a1));
    neg += e0;
    neg += e1;
    pk[j / 2] = bf16x2_bits(e0, e1);
  }
}

// ---- sweep 2 epilogue on 32 columns ---------------------------------------------------------
// PMODE 0: P == 1 ; 1: P from the prob GEMM with GT-new override ; 2: dense P in global memory
// Row constants of sweep 2.  den_ij = exp(s_ij - m_i) + neg_i with exp(.) <= 1; when neg_i >= 4096 (the usual case:
// thousands of negatives with exp(s) up to e^14) x = exp(.)/neg_i <= 2.5e-4 and
//   log2(den) = log2(neg_i) + x log2(e) - O(x^2),   1/den = (1 - x)/neg_i + O(x^2),   |O(x^2)| <= 3e-8,
// so the log and the reciprocal leave the MUFU (one ex2 per pair remains).  Small neg_i takes the exact path.
// In the series path x itself comes out of the ex2: x = 2^(s' ), s' = (s - m) log2(e) - log2(neg_i) = fma(acc, sc, c0),
// then (s - m) log2(e) - log2(den) = s' - x log2(e), Ucoef = w neg_i/den = w (1 - x), and T_i = (1/neg_i) sum Ucoef
// (the 1/neg_i is applied once per row at the end): 11 instructions per pair.
struct RowC {
  float mraw, negi, inv_neg, lneg2, c0;
  bool series;
};

// SERIES is decided per warp (all 32 rows of the warp have neg_i >= 4096), so the pair loop has no divergent branch;
// thr = the row's threshold for the GT-new override of P (min_new for a GT-new row, INT_MAX otherwise).
template <bool FULL, bool SELF, int PMODE, bool SERIES>
__device__ __forceinline__ void sweep2_cols(const uint32_t (&r)[32], const uint32_t (&pr)[32],
                                            const int* __restrict__ lab, int cbase, int nv, int la, int rself,
                                            float sc, const RowC rc, int thr,
                                            const float* __restrict__ dp, float& lacc, float& tacc,
                                            uint32_t (&pk)[16]) {
#pragma unroll
  for (int j4 = 0; j4 < 32; j4 += 4) {
    const int4 l4 = *reinterpret_cast<const int4*>(lab + cbase + j4);
    const int ls[4] = {l4.x, l4.y, l4.z, l4.w};
    float uo[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int col = cbase + j4 + u;
      const float acc = __uint_as_float(r[j4 + u]);
      bool pos = ls[u] == la;
      if (SELF) pos = pos && col != rself;
      if (!FULL) pos = pos && col < nv;
      float pv = 1.f;
      if (PMODE == 1) pv = (ls[u] >= thr) ? 1.f : __uint_as_float(pr[j4 + u]);
      if (PMODE == 2) pv = (FULL || col < nv) ? __ldg(dp + col) : 0.f;
      const float w = pos ? pv : 0.f;
      if (SERIES) {
        const float s2 = fmaf(acc, sc, rc.c0);
        const float x = ex2f(s2);
        lacc = fmaf(w, fmaf(-x, kLog2e, s2), lacc);
        uo[u] = fmaf(-w, x, w);
        tacc += uo[u];  // times 1/neg_i at the end of the sweep
      } else if (PMODE == 3) {  // SupCon statistics over the positive pairs: sum s_ij (log2 units), sum exp(s_ij)
        const float s2 = acc * sc;
        lacc = fmaf(w, s2, lacc);
        tacc = fmaf(w, ex2f(s2), tacc);
        uo[u] = 0.f;
      } else {
        const float sh2 = (acc - rc.mraw) * sc;  // (s - m) * log2(e)
        const float den = ex2f(sh2) + rc.negi;
        lacc = fmaf(w, sh2 - lg2f(den), lacc);
        const float wr = w * rcpf(den);
        tacc += wr;
        uo[u] = wr * rc.negi;
      }
    }
    pk[j4 / 2] = bf16x2_bits(uo[0], uo[1]);
    pk[j4 / 2 + 1] = bf16x2_bits(uo[2], uo[3]);
  }
}

// Sweep-2 fast path: every column of the tile and every row of the warp carry the SAME label (class-sorted tiles make
// this the common case among the tiles sweep 2 visits) and the tile holds neither padding nor the rows themselves:
// every pair is a positive, and the GT-new override of P is one warp-uniform decision (ONES).  No label reads, no
// compares, no selects: ~7 instead of ~11 instructions per pair.
template <bool ONES, bool SERIES>
__device__ __forceinline__ void sweep2_cols_uniform(const uint32_t (&r)[32], const uint32_t (&pr)[32], float sc,
                                                    const RowC rc, float& lacc, float& tacc, uint32_t (&pk)[16]) {
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    float uo[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float acc = __uint_as_float(r[j + u]);
      const float w = ONES ? 1.f : __uint_as_float(pr[j + u]);
      if (SERIES) {
        const float s2 = fmaf(acc, sc, rc.c0);
        const float x = ex2f(s2);
        lacc = fmaf(w, fmaf(-x, kLog2e, s2), lacc);
        uo[u] = fmaf(-w, x, w);
        tacc += uo[u];
      } else {
        const float sh2 = (acc - rc.mraw) * sc;
        const float den = ex2f(sh2) + rc.negi;
        lacc = fmaf(w, sh2 - lg2f(den), lacc);
        const float wr = w * rcpf(den);
        tacc += wr;
        uo[u] = wr * rc.negi;
      }
    }
    pk[j / 2] = bf16x2_bits(uo[0], uo[1]);
  }
}

// ---- sweep 3 (self-contrast losses) on 32 columns ---------------------------------------------
// PixelConLoss v1 and SupConLoss contrast a set of rows with ITSELF and back-propagate through both operands:
// dL/dF = (G + G^T) F / tau with G_ij = dL/ds_ij.  Row i's gradient is therefore sum_j H_ij f_j with H = G + G^T, which
// needs the ROW statistics of pixel i and of pixel j.  They are known after sweeps 1 and 2 (ucd_selfcon_fwd), stored per
// pixel in col_a / col_b / col_c, and this sweep forms H pair by pair and accumulates H F on the tensor cores exactly
// like sweep 1 accumulates V.  e = exp(s_ij):
//   MODE 0 (v1: loss_i = -(1/num_i) sum_j mp_ij [s_ij - log(e + neg_j)]):  a = [num != 0]/num, A = a T (T = sum_j mp_ij /
//           (e + neg_i)), B = neg:   H_ij = (A_i + A_j) e for a negative pair, -a_i [B_i/(e + B_i) + B_j/(e + B_j)] for
//           a positive one (a_j = a_i there: num depends on the label only)
//   MODE 1 (SupCon: loss_i = -a_i [sum_j mp_ij s_ij - num_i (m_i + log D_i)], D_i = sum_{k != i} exp(s_ik - m_i) + 1e-6,
//           a_i = (tau/tau_b)/(num_i + 1e-8) for anchor rows, else 0), A = a num exp(-m)/D:
//           H_ij = (A_i + A_j) e - [positive pair] (a_i + a_j)
// and H_ii = 0.  The common 1/(number of rows in the mean) is applied by ucd_con_bwd.
template <int MODE>
__device__ __forceinline__ void sweep3_cols(const uint32_t (&r)[32], const int* __restrict__ lab, int cbase, int nv, int la,
                                            int rself, float sc, float row_a, float row_b, float row_c,
                                            const float* __restrict__ ca, const float* __restrict__ cb,
                                            uint32_t (&pk)[16]) {
#pragma unroll
  for (int j4 = 0; j4 < 32; j4 += 4) {
    const int4 l4 = *reinterpret_cast<const int4*>(lab + cbase + j4);
    const int ls[4] = {l4.x, l4.y, l4.z, l4.w};
    const float4 a4 = __ldg(reinterpret_cast<const float4*>(ca + cbase + j4));
    const float as[4] = {a4.x, a4.y, a4.z, a4.w};
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(cb + cbase + j4));  // MODE 0: B_j, MODE 1: a_j
    const float bs[4] = {b4.x, b4.y, b4.z, b4.w};
    float h[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int col = cbase + j4 + u;
      const float e = ex2f(__uint_as_float(r[j4 + u]) * sc);
      const bool same = ls[u] == la;
      float v = (row_a + as[u]) * e;
      if (MODE == 0) {
        const float pos = -row_c * (row_b * rcpf(e + row_b) + bs[u] * rcpf(e + bs[u]));
        v = same ? pos : v;
      } else {
        v = same ? v - (row_c + bs[u]) : v;  // a_j differs from a_i when only some rows are anchors ('one' mode)
      }
      h[u] = (col < nv && col != rself) ? v : 0.f;
    }
    pk[j4 / 2] = bf16x2_bits(h[0], h[1]);
    pk[j4 / 2 + 1] = bf16x2_bits(h[2], h[3]);
  }
}

template <int PHASE, int PMODE>
__global__ void __launch_bounds__(kConThreads, 1) con_sweep_kernel(const ConArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];  // no-swizzle operands: 16 B alignment suffices
  __shared__ int s_pre[kMaxChunks + 1];
  __shared__ int s_ncols[kMaxChunks];
  __shared__ uint32_t s_tmem;
  __shared__ uint32_t s_mask[kMaxTilesPerCta / 32];  // bit tt: column tile k0+tt can hold an equal-label pair (or self)

  const long long c_entry = clock64();      // debug trace: CTA set-up and tail cycles
  // Tensor memory: sweep 1: S [0,128) | E (bf16 pairs, two buffers of 64 columns) [128,256) | V [256,512)
  //                sweep 2: S [0,128) | P, later Ucoef [128,256) | U [256,512)
  // ONE S accumulator: it is free again as soon as the epilogue holds the tile in registers (SR), so the S MMAs of
  // tile t+1 run under the epilogue of tile t whatever the V/U MMAs of earlier tiles are doing.  (With E written over
  // S in place, S(t+2) had to wait for V(t): epilogue -> V tail -> S -> epilogue was a two-tile cycle of ~4.9 k clk.)
  // Sweep 2 parks Ucoef in the consumed P columns, so P(t+1) waits for U(t).  (Tried in round 2: a Ucoef tile in shared
  // memory frees the P columns at once but costs one ring slot - with 1.5 tiles in flight every active tile waited for
  // its load: 158 us instead of 125 us per sweep.)
  constexpr int NE = (PHASE != 2) ? 2 : 1;  // E buffers in TMEM (sweep 2 parks Ucoef in the consumed P columns)
  constexpr int NSLOT = (PHASE != 2) ? 5 : 4;  // half-tile slots (sweep 2 keeps 32 KB for the probability operands)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rb = blockIdx.x / a.splits, split = blockIdx.x - rb * a.splits;
  const int n_rows = *a.n_rows;
  if ((long long)rb * 128 >= n_rows) return;  // uniform: nothing to do for this row block

  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + OFF_BAR;
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };

  if (threadIdx.x == 0) {
    int acc = 0;
    for (int c = 0; c < a.n_chunks; ++c) {
      int nc = 0;
      if (c >= a.chunk_lo && c < a.chunk_hi && c != a.chunk_skip) {
        const int* cc = a.chunk_counts + (long long)(c - a.chunk_origin) * (a.chunk_stride ? a.chunk_stride / 4 : 2);
        nc = cc[0] + cc[1];
      }
      s_ncols[c] = nc;
      s_pre[c] = acc;
      acc += (nc + 127) >> 7;
    }
    s_pre[a.n_chunks] = acc;
    mbar_init(BAR(BAR_A), 1);
    for (int i = 0; i < 5; ++i) {
      mbar_init(BAR(BAR_HF + 2 * i), 1);
      mbar_init(BAR(BAR_HF + 2 * i + 1), 1);
      mbar_init(BAR(BAR_HE + i), 1 + kEpiWarps);  // tcgen05.commit + the epilogue warps (they read the tile's labels)
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(BAR(BAR_SF + i), 1);
      mbar_init(BAR(BAR_SE + i), a.need_grad ? 1 : kEpiWarps);  // S buffer free: V MMAs retired / epilogue done
      for (int q = 0; q < 4; ++q) mbar_init(BAR(BAR_EF + 4 * i + q), 4);
    }
    mbar_init(BAR(BAR_PF), 1);
    mbar_init(BAR(BAR_PE), 1);
    mbar_init(BAR(BAR_V), 1);
    mbar_init(BAR(BAR_SR), kEpiWarps);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = s_tmem;

  const int n_total = s_pre[a.n_chunks];
  const int per = (n_total + a.splits - 1) / a.splits;
  const int k0 = split * per;
  const int k1 = min(n_total, k0 + per);
  const int n = max(0, k1 - k0);
  const long long self_tile = a.self_tile0 >= 0 ? a.self_tile0 + rb : -1;  // the anchors' own column tile
  // sweep 2 probability operands: pA (kpad*256 B) stays resident; pC of a tile comes in K chunks of pc_k values
  // (all of it when it fits: kpad <= 64; 16 at a time for kpad = 112, i.e. ADE's 101 old classes).  Beyond 112 old
  // classes (ADE 100-10 / 100-5 from their second step on) pA no longer fits beside a pC chunk: then BOTH operands are
  // streamed, 64 values of K at a time, and pA is re-read per tile (from L2: 256 B per K value, against 64 KB of features)
  const uint32_t pa_bytes = (uint32_t)a.kpad * 256u;
  const bool pa_stream = a.kpad > 112;
  const int pc_k = pa_stream ? 64 : min(a.kpad, (int)((kProbBytes - pa_bytes) / 256u) & ~15);
  const int n_pc = (PHASE == 2 && PMODE == 1) ? (a.kpad + pc_k - 1) / pc_k : 0;
  const uint32_t off_pc = OFF_PA + (pa_stream ? 64u * 256u : pa_bytes);
  // Sweep 2 only touches pairs with equal labels (w_ij = 0 otherwise): a column tile whose label range misses the
  // row block's range contributes nothing and is skipped by all three roles (class-sorted tiles make this common).
  // Label-overlap mask of this CTA's column tiles, evaluated once by all threads (the range lookups are L2
  // round trips: doing them per tile inside the role loops would put ~1.5k cycles of latency on every tile).
  // Sweep 2 only walks the set bits (w_ij = 0 for unequal labels); sweep 1 uses the clear bits to pick the
  // all-negative fast path.  Class-sorted tiles make clear bits the common case.
  {
    const int row_lo = __ldg(a.row_range + 2 * rb), row_hi = __ldg(a.row_range + 2 * rb + 1);
    for (int base = 0; base < n; base += kConThreads) {
      const int tt = base + (int)threadIdx.x;
      bool ov = false;
      if (tt < n) {
        const TileLoc loc = locate_tile(k0 + tt, s_pre, s_ncols, a.n_chunks, a.chunk_tiles);
        const int* tr = reinterpret_cast<const int*>(reinterpret_cast<const uint8_t*>(a.tile_range) +
                                                     tile_off(loc, 8, a.chunk_tiles, a.chunk_stride, a.chunk_origin));
        const int lo = __ldg(tr), hi = __ldg(tr + 1);
        ov = loc.gtile == self_tile || !(hi < row_lo || lo > row_hi);
      }
      const unsigned bits = __ballot_sync(0xffffffffu, ov);
      if (lane == 0 && base + warp * 32 < n) s_mask[(base >> 5) + warp] = bits;
    }
    __syncthreads();
  }
  // next tile index >= tt that this sweep has to process (sweep 1: every tile; sweep 2: next set mask bit)
  auto next_active = [&](int tt) -> int {
    if (PHASE != 2) return tt;
    while (tt < n) {
      const uint32_t bits = s_mask[tt >> 5] >> (tt & 31);
      if (bits) return tt + __ffs(bits) - 1;
      tt = (tt | 31) + 1;
    }
    return n;
  };

  // The three issuing roles run WARP-UNIFORM: all 32 lanes walk the tile loop and wait on the barriers, and the
  // uniform-datapath instructions (bulk copies, tcgen05.mma, tcgen05.commit) sit in elect_one_sync() blocks, so that
  // ptxas emits them back to back from uniform registers (see umma.cuh; `if (lane == 0)` costs an ELECT/BRA.U.ANY
  // loop around every one of them).
  if (warp == 0) {
    // ===================== producer: bulk async copies =====================
    if (n > 0) {
      const uint8_t* ft = reinterpret_cast<const uint8_t*>(a.feat_tiles);
      const uint8_t* pt = reinterpret_cast<const uint8_t*>(a.prob_tiles);
      const uint8_t* rft = reinterpret_cast<const uint8_t*>(a.row_feat);
      const uint8_t* rpt = reinterpret_cast<const uint8_t*>(a.row_prob);
      const uint32_t pbytes = pa_bytes;
      if (elect_one_sync()) {
        mbar_arrive_expect_tx(BAR(BAR_A), kTileBytes + ((PHASE == 2 && PMODE == 1 && !pa_stream) ? pbytes : 0u));
#pragma unroll
        for (int q = 0; q < 4; ++q)
          bulk_g2s(sbase + OFF_A + q * 16384u, rft + (size_t)rb * kTileBytes + q * 16384u, 16384u, BAR(BAR_A));
        if (PHASE == 2 && PMODE == 1 && !pa_stream)
          bulk_g2s(sbase + OFF_PA, rpt + (size_t)rb * pbytes, pbytes, BAR(BAR_A));
      }
      __syncwarp();
      long long w_ce = 0, w_pe = 0;
      const long long c_start = clock64();
      int t = 0;
      Ring<NSLOT> ring;
      TileCursor cur;
      cur.init(s_pre, s_ncols, a.n_chunks, a.chunk_tiles);
      for (int tt = next_active(0); tt < n; tt = next_active(tt + 1)) {
        const TileLoc loc = cur.seek(k0 + tt);
        const int lb = t % 3;  // label buffer: reloaded for tile t+3, whose first slot is freed after tile t (or t+1)
#pragma unroll
        for (int fh = 0; fh < 2; ++fh) {
          mbar_wait_t(BAR(BAR_HE + ring.slot), ring.par ^ 1u, w_ce);
          if (elect_one_sync()) {
            const uint32_t dst = sbase + OFF_C + (uint32_t)ring.slot * kSlotBytes;
            const uint8_t* src = ft + tile_off(loc, kTileBytes, a.chunk_tiles, a.chunk_stride, a.chunk_origin) +
                                 (size_t)fh * kSlotBytes;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const uint32_t bq = BAR(BAR_HF + 2 * ring.slot + q);
              const bool with_labels = fh == 0 && q == 0;
              mbar_arrive_expect_tx(bq, 16384u + (with_labels ? 512u : 0u));
              bulk_g2s(dst + q * 16384u, src + q * 16384u, 16384u, bq);
              if (with_labels)
                bulk_g2s(sbase + OFF_LAB + lb * 512u, reinterpret_cast<const uint8_t*>(a.lab_tiles) +
                                                          tile_off(loc, 512, a.chunk_tiles, a.chunk_stride, a.chunk_origin),
                         512u, bq);
            }
          }
          __syncwarp();
          ring.next();
        }
        for (int c = 0; c < n_pc; ++c) {  // column probabilities, one K chunk at a time through a single buffer
          const int u = t * n_pc + c;
          const uint32_t kb = (uint32_t)min(pc_k, a.kpad - c * pc_k) * 256u;
          mbar_wait_t(BAR(BAR_PE), (u & 1) ^ 1, w_pe);
          if (elect_one_sync()) {
            mbar_arrive_expect_tx(BAR(BAR_PF), pa_stream ? 2u * kb : kb);
            bulk_g2s(sbase + off_pc, pt + tile_off(loc, pbytes, a.chunk_tiles, a.chunk_stride, a.chunk_origin) +
                                         (size_t)c * pc_k * 256u, kb, BAR(BAR_PF));
            if (pa_stream)  // the same K chunk of the row probabilities
              bulk_g2s(sbase + OFF_PA, rpt + (size_t)rb * pbytes + (size_t)c * pc_k * 256u, kb, BAR(BAR_PF));
          }
          __syncwarp();
        }
        ++t;
      }
      if (a.trace && lane == 0) {
        long long* tr = a.trace + (size_t)blockIdx.x * 16;
        tr[0] = clock64() - c_start, tr[1] = w_ce, tr[2] = w_pe, tr[3] = t;
      }
    }
  } else if (warp == 1) {
    // ===================== S issuer: S = A C^T (and P = pA pC^T in sweep 2) =====================
    // S and V/U are issued by two different warps so that neither waits behind the other's barriers.
    if (n > 0) {
      constexpr uint32_t idesc_s = umma_idesc(128, 128, 0, 0);   // A K-major, B K-major
      const uint32_t tS = tmem, tP = tmem + 128;
      const uint64_t adesc0 = umma_desc(sbase + OFF_A, kChunkB, 128);
      const uint64_t cdesc0 = umma_desc(sbase + OFF_C, kChunkB, 128);
      const uint64_t padesc0 = umma_desc(sbase + OFF_PA, kChunkB, 128);
      const uint64_t pcdesc0 = umma_desc(sbase + off_pc, kChunkB, 128);
      mbar_wait(BAR(BAR_A), 0);
      long long c_idle = 0;
      const long long c_start = clock64();
      int t = 0;
      Ring<NSLOT> ring;
      for (int tt = next_active(0); tt < n; tt = next_active(tt + 1)) {
        constexpr int sb = 0;
        const int slot_a = ring.slot;  // the tile's first slot (features 0-127); the second one follows in the ring
        // S may be overwritten as soon as the epilogue holds the previous tile in registers
        mbar_wait_t(BAR(BAR_SR), (t & 1) ^ 1, c_idle);
#pragma unroll
        for (int q = 0; q < 4; ++q) {  // 4 K steps per landed 16 KB quarter of the column tile (two per slot)
          const int hq = q & 1;
          mbar_wait_t(BAR(BAR_HF + 2 * ring.slot + hq), ring.par, c_idle);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint64_t cdesc = umma_desc_adv(cdesc0, (uint32_t)ring.slot * kSlotBytes + (uint32_t)hq * 16384u);
            const uint64_t adesc = umma_desc_adv(adesc0, (uint32_t)q * 16384u);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_bf16(tS + sb * 128, umma_desc_adv(adesc, ks * 2 * kChunkB), umma_desc_adv(cdesc, ks * 2 * kChunkB),
                        idesc_s, (q > 0 || ks > 0) ? 1u : 0u);
            if (q == 3 && PHASE != 2) {
              umma_commit(BAR(BAR_SF + sb));
              if (!a.need_grad) {  // no V pass: the slots are free once S is done
                umma_commit(BAR(BAR_HE + slot_a));
                umma_commit(BAR(BAR_HE + ring.slot));
              }
            }
          }
          __syncwarp();
          if (hq == 1) ring.next();
        }
        const int slot_b = (slot_a + 1 == NSLOT) ? 0 : slot_a + 1;
        if (PHASE == 2) {
          // the P columns (Ucoef of the previous tile lives there, whatever PMODE is) are free once its U MMAs
          // retired: the epilogue of this tile must not get SF before that
          mbar_wait_t(BAR(BAR_SE), (t & 1) ^ 1, c_idle);
          tc_fence_after();
          if (n_pc == 0) {
            if (elect_one_sync()) {
              umma_commit(BAR(BAR_SF + sb));
              if (!a.need_grad) {
                umma_commit(BAR(BAR_HE + slot_a));
                umma_commit(BAR(BAR_HE + slot_b));
              }
            }
            __syncwarp();
          }
          for (int c = 0; c < n_pc; ++c) {  // P = pA pC^T accumulated over the K chunks of pC
            const int u = t * n_pc + c;
            mbar_wait_t(BAR(BAR_PF), u & 1, c_idle);
            tc_fence_after();
            const int ksteps = min(pc_k, a.kpad - c * pc_k) >> 4;
            if (elect_one_sync()) {
              for (int ks = 0; ks < ksteps; ++ks)
                umma_bf16(tP, umma_desc_adv(padesc0, (uint32_t)((pa_stream ? 0 : c * (pc_k >> 3)) + ks * 2) * kChunkB),
                          umma_desc_adv(pcdesc0, ks * 2 * kChunkB), idesc_s, (c > 0 || ks > 0) ? 1u : 0u);
              umma_commit(BAR(BAR_PE));
              if (c == n_pc - 1) {
                umma_commit(BAR(BAR_SF + sb));
                if (!a.need_grad) {
                  umma_commit(BAR(BAR_HE + slot_a));
                  umma_commit(BAR(BAR_HE + slot_b));
                }
              }
            }
            __syncwarp();
          }
        }
        ++t;
      }
      if (!a.need_grad) {
        if (elect_one_sync()) umma_commit(BAR(BAR_V));
        __syncwarp();
      }
      if (a.trace && lane == 0) {
        long long* tr = a.trace + (size_t)blockIdx.x * 16;
        tr[4] = clock64() - c_start, tr[5] = c_idle, tr[6] = t;
      }
    }
  } else if (warp == 2) {
    // ===================== V/U issuer: acc += E x C with E (bf16) read from tensor memory ============
    if (n > 0 && a.need_grad) {
      constexpr uint32_t idesc_v = umma_idesc(128, 128, 0, 1);   // A from TMEM, B MN-major: one feature half (slot)
      const uint32_t tV = tmem + 256;
      const uint64_t vdesc0 = umma_desc(sbase + OFF_C, 128, kChunkB);
      long long c_idle = 0;
      const long long c_start = clock64();
      int t = 0;
      int slot_a = 0;
      for (int tt = next_active(0); tt < n; tt = next_active(tt + 1)) {
        const int eb = t % NE;
        const int slot_b = (slot_a + 1 == NSLOT) ? 0 : slot_a + 1;
#pragma unroll
        for (int u = 0; u < 4; ++u) {  // (chunk 0, half 0), (chunk 0, half 1), (chunk 1, half 0), (chunk 1, half 1)
          const int cc = u >> 1, h = u & 1;
          mbar_wait_t(BAR(BAR_EF + (eb * 2 + h) * 2 + cc), (t / NE) & 1, c_idle);
          tc_fence_after();
          // 16 columns of packed bf16 pairs = 32 K values: E buffer eb (sweep 1), Ucoef over P (sweep 2)
          const uint32_t te = tmem + 128 + (PHASE != 2 ? eb * 64 + h * 32 : h * 64) + cc * 16;
          if (elect_one_sync()) {
            const uint32_t rowoff = (uint32_t)(h * 64 + cc * 32) * 16u;
            const uint64_t vda = umma_desc_adv(vdesc0, (uint32_t)slot_a * kSlotBytes + rowoff);
            const uint64_t vdb = umma_desc_adv(vdesc0, (uint32_t)slot_b * kSlotBytes + rowoff);
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              const uint32_t acc = (t > 0 || u > 0 || kk > 0) ? 1u : 0u;
              umma_bf16_ts(tV, te + kk * 8, umma_desc_adv(vda, (uint32_t)kk * 256u), idesc_v, acc);         // features 0-127
              umma_bf16_ts(tV + 128, te + kk * 8, umma_desc_adv(vdb, (uint32_t)kk * 256u), idesc_v, acc);   // 128-255
            }
            if (u == 3) {
              umma_commit(BAR(BAR_HE + slot_a));  // tile t no longer needs its two slots ...
              umma_commit(BAR(BAR_HE + slot_b));
              umma_commit(BAR(BAR_SE + eb));      // ... nor its E buffer (sweep 2: the P columns)
            }
          }
          __syncwarp();
        }
        slot_a = (slot_b + 1 == NSLOT) ? 0 : slot_b + 1;
        ++t;
      }
      if (elect_one_sync()) umma_commit(BAR(BAR_V));
      __syncwarp();
      if (a.trace && lane == 0) {
        long long* tr = a.trace + (size_t)blockIdx.x * 16;
        tr[12] = clock64() - c_start, tr[13] = c_idle, tr[14] = t;
      }
    }
  } else {
    // ===================== epilogue: one thread per row =====================
    // warps 3-6 own columns [0,64) of every tile (E half 0), warps 7-10 columns [64,128) (half 1);
    // within a half, warp w reads TMEM lanes 32*(w%4).. (hardware restriction) = rows of the block.
    const int half = (warp - 3) >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;  // row within the block == TMEM lane
    const long long grow = (long long)rb * 128 + r;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const int la = (grow < n_rows) ? __ldg(a.row_lab + (size_t)rb * 128 + r) : -2;
    const float sc = a.inv_tau * kLog2e;
    float mx = -3.0e38f, neg = 0.f, num = 0.f;   // sweep 1
    float lacc = 0.f, tacc = 0.f;                // sweep 2
    RowC rc = {0.f, 0.f, 0.f, 0.f, 0.f, false};
    int thr = 0x7fffffff;
    bool warp_series = false;
    float row_a = 0.f, row_b = 0.f, row_c = 0.f;  // sweep 3: this pixel's coefficients
    if (PHASE == 3 && grow < n_rows) row_a = a.col_a[grow], row_b = a.col_b[grow], row_c = a.col_c[grow];
    if (PHASE == 2) {
      rc.mraw = a.shift ? a.stats[grow] : 0.f;
      rc.negi = a.stats[a.rows_pad + grow];
      rc.series = PMODE != 3 && rc.negi >= 4096.f;
      rc.inv_neg = rc.series ? 1.f / rc.negi : 0.f;
      rc.lneg2 = rc.series ? log2f(rc.negi) : 0.f;
      rc.c0 = -fmaf(rc.mraw, sc, rc.lneg2);
      if (PMODE == 1) {
        int min_new = 0x7fffffff;  // global GT-new threshold = minimum over every rank's chunk header
        for (int c = 0; c < (a.chunk_stride ? a.n_chunks : 1); ++c)
          min_new = min(min_new, __ldg(a.min_new + (long long)(c - a.chunk_origin) * (a.chunk_stride / 4)));
        if (la >= min_new) thr = min_new;  // GT-new row: P = 1 against GT-new columns (loss.py:385-393)
      }
      warp_series = __all_sync(0xffffffffu, rc.series);
      rc.series = warp_series;  // rows of a mixed warp all take the exact path
    }
    int t = 0;  // number of active tiles processed so far (drives buffer / parity bookkeeping)
    int slot_a = 0;  // first ring slot of the current tile
    long long w_sf = 0, w_ee = 0;  // w_ee: wait for a free E buffer (sweep 1)
    const long long c_start = clock64();
    TileCursor cur;
    cur.init(s_pre, s_ncols, a.n_chunks, a.chunk_tiles);
    uint32_t mword = (PHASE == 1 && n > 0) ? s_mask[0] : 0u;  // sweep 1: overlap bits of tiles [32w, 32w+32) in a register
    for (int tt = next_active(0); tt < n; tt = next_active(tt + 1)) {
      const TileLoc loc = cur.seek(k0 + tt);
      if (PHASE == 1 && (tt & 31) == 0 && tt > 0) mword = s_mask[tt >> 5];
      constexpr int sb = 0;
      const int eb = t % NE;
      const int slot_b = (slot_a + 1 == NSLOT) ? 0 : slot_a + 1;
      const bool full = loc.nvalid == 128;
      const bool self = loc.gtile == self_tile;
      const int* lab = reinterpret_cast<const int*>(smem + OFF_LAB + (t % 3) * 512);
      const float* dp = (PMODE == 2) ? a.dense_p + (size_t)min(grow, (long long)n_rows - 1) * a.ldp + loc.dcol0 : nullptr;
      const bool all_neg = PHASE == 1 && full && !((mword >> (tt & 31)) & 1u);
      mbar_wait_t(BAR(BAR_SF + sb), t & 1, w_sf);
      tc_fence_after();
      // E / Ucoef sub-tile hand-off to the MMA warp: 32 packed bf16 of this row go to k-chunks (cc&1)*4..+3
      // E / Ucoef hand-off to the MMA warp: the 32 bf16 of this chunk overwrite the first columns of the thread's
      // own (already consumed) S range in tensor memory; the V/U MMA reads its A operand from there.
      auto emit = [&](int cc, const uint32_t (&pk)[16]) {  // cc = chunk 0/1 within this thread's column half
        if (!a.need_grad) return;
        tmem_st16(tmem + lane_addr + 128 + (PHASE != 2 ? eb * 64 + half * 32 : half * 64) + cc * 16, pk);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(BAR(BAR_EF + (eb * 2 + half) * 2 + cc));
      };
      const int c0 = half * 64;  // first column of this thread's half
      if (PHASE != 2) {
        // software-pipelined TMEM reads: the second chunk is in flight while the first is processed
        uint32_t r0[32], r1[32];
        auto proc = [&](int cc, const uint32_t (&rv)[32]) {
          uint32_t pk[16];
          if (PHASE == 3)
            sweep3_cols<PMODE>(rv, lab, c0 + cc * 32, loc.nvalid, la, self ? r : -1, sc, row_a, row_b, row_c,
                               a.col_a + loc.dcol0, (PMODE == 0 ? a.col_b : a.col_c) + loc.dcol0, pk);
          else if (all_neg)
            sweep1_cols_neg(rv, sc, mx, neg, pk);
          else if (full && !self)
            sweep1_cols<true, false>(rv, lab, c0 + cc * 32, 128, la, r, sc, mx, neg, num, pk);
          else
            sweep1_cols<false, true>(rv, lab, c0 + cc * 32, loc.nvalid, la, self ? r : -1, sc, mx, neg, num, pk);
          emit(cc, pk);
        };
        const uint32_t tb = tmem + lane_addr + c0;
        tmem_ld32(tb, r0);
        tmem_ld32(tb + 32, r1);
        if (a.need_grad) {  // E buffer eb is free once the V MMAs of tile t-2 have retired (rarely a real wait; the
          mbar_wait_t(BAR(BAR_SE + eb), ((t >> 1) & 1) ^ 1, w_ee);  // barrier round trip hides under the loads)
        }
        tmem_ld_wait();
        tmem_ld_fence(r0);
        tmem_ld_fence(r1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(BAR(BAR_SR));  // S of this tile is in registers: the next tile's S MMAs may start
        tc_fence_after();
        proc(0, r0);
        proc(1, r1);
      } else {
        // uniform tile: the 32 row labels of the warp are one label and all 128 column labels equal it.  Lane k
        // compares only columns 4k..4k+3, so the row labels must be checked on their own: a warp with rows a|b split
        // at lane K against a tile with columns a|b split at 4K passes the column compare alone.  Rows past n_rows
        // (la = -2) never pass.
        bool uniform = false;
        if (PMODE != 2 && PMODE != 3 && full && !self) {
          const int4 l4 = *reinterpret_cast<const int4*>(lab + lane * 4);
          uniform = __all_sync(0xffffffffu, la == __shfl_sync(0xffffffffu, la, 0) && l4.x == la && l4.y == la &&
                                                l4.z == la && l4.w == la);
        }
        const bool ones = PMODE == 0 || la >= thr;  // warp-uniform when `uniform` (same la, hence same thr, in every lane)
#pragma unroll 1
        for (int cc = 0; cc < 2; ++cc) {
          uint32_t rv[32], pv[32], pk[16];
          tmem_ld32(tmem + lane_addr + sb * 128 + c0 + cc * 32, rv);
          if (PMODE == 1) tmem_ld32(tmem + lane_addr + 128 + c0 + cc * 32, pv);
          tmem_ld_wait();
          tmem_ld_fence(rv);
          if (PMODE == 1) tmem_ld_fence(pv);
          if (cc == 1) {  // S (and P) of this tile are in registers: the next tile's S and P MMAs may start
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR(BAR_SR));
          }
          if (uniform) {
            if (ones) {
              if (warp_series)
                sweep2_cols_uniform<true, true>(rv, pv, sc, rc, lacc, tacc, pk);
              else
                sweep2_cols_uniform<true, false>(rv, pv, sc, rc, lacc, tacc, pk);
            } else {
              if (warp_series)
                sweep2_cols_uniform<false, true>(rv, pv, sc, rc, lacc, tacc, pk);
              else
                sweep2_cols_uniform<false, false>(rv, pv, sc, rc, lacc, tacc, pk);
            }
          } else if (full && !self) {
            if (warp_series)
              sweep2_cols<true, false, PMODE, true>(rv, pv, lab, c0 + cc * 32, 128, la, r, sc, rc, thr, dp, lacc, tacc, pk);
            else
              sweep2_cols<true, false, PMODE, false>(rv, pv, lab, c0 + cc * 32, 128, la, r, sc, rc, thr, dp, lacc, tacc, pk);
          } else {
            if (warp_series)
              sweep2_cols<false, true, PMODE, true>(rv, pv, lab, c0 + cc * 32, loc.nvalid, la, self ? r : -1, sc, rc,
                                                    thr, dp, lacc, tacc, pk);
            else
              sweep2_cols<false, true, PMODE, false>(rv, pv, lab, c0 + cc * 32, loc.nvalid, la, self ? r : -1, sc, rc,
                                                     thr, dp, lacc, tacc, pk);
          }
          emit(cc, pk);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PHASE == 2 && !a.need_grad) mbar_arrive(BAR(BAR_SE));
        mbar_arrive(BAR(BAR_HE + slot_a));  // this warp no longer reads the tile's labels
        mbar_arrive(BAR(BAR_HE + slot_b));
      }
      slot_a = (slot_b + 1 == NSLOT) ? 0 : slot_b + 1;
      ++t;
    }
    if (a.trace && warp == 3 && lane == 0) {  // one representative epilogue thread
      long long* tr = a.trace + (size_t)blockIdx.x * 16;
      tr[8] = clock64() - c_start, tr[9] = w_sf, tr[10] = w_ee, tr[11] = t;
      tr[7] = c_start - c_entry;
    }
    const long long c_tail = clock64();
    // ---- per-row outputs: the two column halves of a row combine through shared memory ----
    if (a.need_grad && t > 0) {  // all MMAs retired: accumulator final, E buffers free for reuse below
      mbar_wait(BAR(BAR_V), 0);
      tc_fence_after();
    }
    // [128][3] scratch in C stage 0: every tile load has landed and every MMA that reads the stages has retired
    // by now.  (NOT the probability region: with no active tile the row-probability copy may still be in flight.)
    if (PHASE == 2 && rc.series) tacc *= rc.inv_neg;  // the series path accumulated sum_j Ucoef_ij = neg_i T_i
    float* comb = reinterpret_cast<float*>(smem + OFF_C);
    if (PHASE != 3 && half == 1) {
      comb[r * 3 + 0] = PHASE == 1 ? mx : lacc;
      comb[r * 3 + 1] = PHASE == 1 ? neg : tacc;
      comb[r * 3 + 2] = num;
    }
    asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
    if (PHASE != 3 && half == 0) {
      if (PHASE == 1) {
        const size_t slot = (size_t)(split + a.split_base);
        a.stats_part[slot * 3 * a.rows_pad + grow] = fmaxf(mx, comb[r * 3 + 0]);
        a.stats_part[slot * 3 * a.rows_pad + a.rows_pad + grow] = neg + comb[r * 3 + 1];
        a.stats_part[slot * 3 * a.rows_pad + 2 * a.rows_pad + grow] = num + comb[r * 3 + 2];
      } else {
        a.loss_part[(size_t)split * 2 * a.rows_pad + grow] = (lacc + comb[r * 3 + 0]) * kLn2;
        a.loss_part[(size_t)split * 2 * a.rows_pad + a.rows_pad + grow] = tacc + comb[r * 3 + 1];
      }
    }
    if (a.need_grad) {  // each half writes 128 of the 256 accumulator columns of its rows
      // tcgen05.ld hands a thread 32 consecutive columns of ITS row; stored directly, one instruction would touch 32
      // different 128-byte lines with 16 bytes each.  A per-warp [32][36] transposition buffer in the (now idle) C stage
      // turns that into 4 full lines per instruction.
      float* xp = reinterpret_cast<float*>(smem + OFF_C + 4096) + (size_t)(warp - 3) * (32 * 36);
      const size_t prow0 = (size_t)(split + (PHASE != 2 ? a.split_base : 0)) * a.rows_pad + (size_t)rb * 128 +
                           quarter * 32;  // first row of this warp
      float* dstw = a.acc_part + prow0 * 256 + half * 128;
      const int orow = lane >> 3, ocol = (lane & 7) * 4;
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        if (t > 0) {
          uint32_t rv[32];
          tmem_ld32(tmem + lane_addr + 256 + half * 128 + cc * 32, rv);
          tmem_ld_wait();
          tmem_ld_fence(rv);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            *reinterpret_cast<float4*>(xp + lane * 36 + 4 * k) =
                make_float4(__uint_as_float(rv[4 * k]), __uint_as_float(rv[4 * k + 1]), __uint_as_float(rv[4 * k + 2]),
                            __uint_as_float(rv[4 * k + 3]));
          __syncwarp();
        }
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int row = it * 4 + orow;
          const float4 v = t > 0 ? *reinterpret_cast<const float4*>(xp + row * 36 + ocol) : make_float4(0.f, 0.f, 0.f, 0.f);
          *reinterpret_cast<float4*>(dstw + (size_t)row * 256 + cc * 32 + ocol) = v;
        }
        __syncwarp();
      }
    }
    tc_fence_before();
    if (a.trace && warp == 3 && lane == 0) a.trace[(size_t)blockIdx.x * 16 + 15] = clock64() - c_tail;
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// combine sweep-1 partials over splits: stats[0]=row max (raw dot), [1]=neg, [2]=num
__global__ void con_combine_kernel(const float* __restrict__ part, int splits, long long rows_pad,
                                   float* __restrict__ stats) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows_pad) return;
  float m = -3.0e38f, neg = 0.f, num = 0.f;
  for (int s = 0; s < splits; ++s) {
    const float* p = part + (size_t)s * 3 * rows_pad;
    m = fmaxf(m, p[i]);
    neg += p[rows_pad + i];
    num += p[2 * rows_pad + i];
  }
  stats[i] = m;
  stats[rows_pad + i] = neg;
  stats[2 * rows_pad + i] = num;
}

// finalize: per-row loss terms, unit gradient, per-block partial sums.  block = 4 rows x 64 threads, a thread owns
// one float4 of its row: splits + splits2 independent 16 B streaming loads in flight per thread.
__global__ void __launch_bounds__(256)
con_finalize_kernel(const float* __restrict__ stats, const float* __restrict__ loss_part,
                    const float* __restrict__ v_part, const float* __restrict__ u_part, int splits, int splits2,
                    long long rows_pad, const int* __restrict__ n_rows_p, float inv_tau,
                    int need_grad, float* __restrict__ grad_unit, float* __restrict__ block_part) {
  const int n_rows = *n_rows_p;
  const int sub = threadIdx.x >> 6, q = threadIdx.x & 63;
  float lsum = 0.f, lcnt = 0.f;
#pragma unroll 2  // two rows' loads in flight: 30 -> 27 us at the bench size (6.3 TB/s, the read ceiling)
  for (long long row = (long long)blockIdx.x * 4 + sub; row < n_rows; row += (long long)gridDim.x * 4) {
    const float num = stats[2 * rows_pad + row];
    float L = 0.f, T = 0.f;
    for (int s = 0; s < splits2; ++s) {
      L += loss_part[(size_t)s * 2 * rows_pad + row];
      T += loss_part[(size_t)s * 2 * rows_pad + rows_pad + row];
    }
    const bool valid = num != 0.f;
    if (need_grad) {
      float4 V = make_float4(0.f, 0.f, 0.f, 0.f), U = V;
#pragma unroll 4
      for (int s = 0; s < splits; ++s) {
        const float4 t = __ldcs(reinterpret_cast<const float4*>(v_part + ((size_t)s * rows_pad + row) * 256) + q);
        V.x += t.x, V.y += t.y, V.z += t.z, V.w += t.w;
      }
#pragma unroll 4
      for (int s = 0; s < splits2; ++s) {
        const float4 t = __ldcs(reinterpret_cast<const float4*>(u_part + ((size_t)s * rows_pad + row) * 256) + q);
        U.x += t.x, U.y += t.y, U.z += t.z, U.w += t.w;
      }
      const float k = valid ? inv_tau / num : 0.f;
      float4 g;
      g.x = valid ? k * (T * V.x - U.x) : 0.f;
      g.y = valid ? k * (T * V.y - U.y) : 0.f;
      g.z = valid ? k * (T * V.z - U.z) : 0.f;
      g.w = valid ? k * (T * V.w - U.w) : 0.f;
      reinterpret_cast<float4*>(grad_unit + (size_t)row * 256)[q] = g;
    }
    if (q == 0 && valid) {
      lsum += -L / num;
      lcnt += 1.f;
    }
  }
  __shared__ float sh[2][4];
  if (q == 0) sh[0][sub] = lsum, sh[1][sub] = lcnt;
  __syncthreads();
  if (threadIdx.x == 0) {  // fixed order
    block_part[blockIdx.x] = (sh[0][0] + sh[0][1]) + (sh[0][2] + sh[0][3]);
    block_part[gridDim.x + blockIdx.x] = (sh[1][0] + sh[1][1]) + (sh[1][2] + sh[1][3]);
  }
}

// out = {sum of row losses, number of valid rows, their ratio (the loss; NaN when no row is valid, like the reference)}
__global__ void con_reduce_out_kernel(const float* __restrict__ block_part, int nblk, float* __restrict__ out) {
  __shared__ float red[32];
  __shared__ float res[2];
  for (int k = 0; k < 2; ++k) {
    float acc = 0.f;
    for (int i = threadIdx.x; i < nblk; i += blockDim.x) acc += block_part[(size_t)k * nblk + i];
    const float r = block_sum(acc, red);
    if (threadIdx.x == 0) out[k] = r, res[k] = r;
  }
  if (threadIdx.x == 0) out[2] = res[0] / res[1];
}

__global__ void con_bwd_kernel(const float* __restrict__ grad_unit, const float* __restrict__ out,
                               const float* __restrict__ g_scalar, float g_mul, const int* __restrict__ n_rows_p,
                               const int* __restrict__ row_ref, float* __restrict__ d_anchor, long long max_rows) {
  const long long n_rows = min((long long)*n_rows_p, max_rows);
  const float coef = (out[1] > 0.f) ? g_scalar[0] * g_mul / out[1] : 0.f;
  const long long n4 = n_rows * 64;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 g = reinterpret_cast<const float4*>(grad_unit)[i];
    g.x *= coef, g.y *= coef, g.z *= coef, g.w *= coef;
    const long long row = i >> 6;
    const long long dst = row_ref ? (long long)row_ref[row] : row;  // tile (class-sorted) row -> reference row
    reinterpret_cast<float4*>(d_anchor)[dst * 64 + (i & 63)] = g;
  }
}

// Self-contrast losses, between sweep 2 and sweep 3: per-pixel coefficients of sweep3_cols, the per-row loss terms and
// their per-block partial sums.  mode 0 = PixelConLoss v1, 1 = SupConLoss (n_anchor: rows that are anchors, the first
// ones; kappa = temperature / base_temperature).  stats = {raw row max, neg, num} of sweep 1; loss_part = sweep 2's
// {L_i, T_i} (v1: unshifted denominator) or {sum_pos s_ij, sum_pos exp(s_ij)} (SupCon).
__global__ void __launch_bounds__(256)
selfcon_rowcoef_kernel(const float* __restrict__ stats, const float* __restrict__ loss_part, int splits2,
                       long long rows_pad, long long n, long long n_anchor, int mode, float inv_tau, float kappa,
                       float* __restrict__ col_a, float* __restrict__ col_b, float* __restrict__ col_c,
                       float* __restrict__ block_part) {
  float lsum = 0.f, lcnt = 0.f;
  for (long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x; row < rows_pad;
       row += (long long)gridDim.x * blockDim.x) {
    float ca = 0.f, cb = 0.f, cc = 0.f;
    if (row < n) {
      const float neg = stats[rows_pad + row], num = stats[2 * rows_pad + row];
      float p0 = 0.f, p1 = 0.f;
      for (int s = 0; s < splits2; ++s) {
        p0 += loss_part[(size_t)s * 2 * rows_pad + row];
        p1 += loss_part[(size_t)s * 2 * rows_pad + rows_pad + row];
      }
      if (mode == 0) {
        const bool valid = num != 0.f;
        cc = valid ? 1.f / num : 0.f;
        ca = cc * p1;
        cb = neg;
        if (valid) lsum += -p0 / num, lcnt += 1.f;
      } else {
        const float m = stats[row] * inv_tau;                      // max_j s_ij, the row itself included
        const float em = __expf(-m);
        const float D = (neg + p1) * em + 1e-6f;                   // sum_{k != i} exp(s_ik - m) + 1e-6 (loss_new.py:340)
        cc = row < n_anchor ? kappa / (num + 1e-8f) : 0.f;        // fp32 like the reference's float mask (loss_new.py:345)
        ca = cc * num * em / D;
        if (row < n_anchor) lsum += -cc * (p0 - num * (m + __logf(D))), lcnt += 1.f;
      }
    }
    col_a[row] = ca, col_b[row] = cb, col_c[row] = cc;
  }
  __shared__ float red[32];
  const float r0 = block_sum(lsum, red);
  const float r1 = block_sum(lcnt, red);
  if (threadIdx.x == 0) block_part[blockIdx.x] = r0, block_part[gridDim.x + blockIdx.x] = r1;
}

// unit gradient of the self-contrast losses: (1/tau) * sum over the column splits of sweep 3's partial products
__global__ void __launch_bounds__(256)
selfcon_grad_kernel(const float* __restrict__ v_part, int splits, long long rows_pad, long long n, float inv_tau,
                    float* __restrict__ grad_unit) {
  const long long n4 = n * 64;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < splits; ++s) {
      const float4 t = __ldcs(reinterpret_cast<const float4*>(v_part + (size_t)s * rows_pad * 256) + i);
      acc.x += t.x, acc.y += t.y, acc.z += t.z, acc.w += t.w;
    }
    reinterpret_cast<float4*>(grad_unit)[i] = make_float4(acc.x * inv_tau, acc.y * inv_tau, acc.z * inv_tau, acc.w * inv_tau);
  }
}

constexpr int kFinalizeBlocks = kNumSMs * 4;
#ifdef UCD_DEBUG_KNOBS
static long long* g_trace = nullptr;  // debug builds only (ucd_con_debug_trace)
#endif

struct ConPlan {
  int splits;        // column splits of sweep 1 (one launch over all chunks), or of its REMOTE part (two-part run)
  int splits_local;  // two-part run: column splits of the launch over the local chunk (0 = single launch)
  int splits2;       // column splits of sweep 2 (few active tiles per CTA: fewer, longer CTAs amortise the fixed cost)
  long long rows_pad;
  size_t off_stats_part, off_stats, off_loss_part, off_v, off_u, off_block, total;
  int splits1_total() const { return splits + splits_local; }
};

// number of column splits that best fills the SMs with `row_tiles` row blocks without tiny per-CTA column ranges
static int choose_splits(long long row_tiles, long long col_tiles) {
  int best = 1;
  double best_eff = 0.0;
  for (int s = 1; s <= 16; ++s) {
    if (s > 1 && col_tiles / s < 4) break;
    const long long ctas = row_tiles * s;
    const long long waves = (ctas + kNumSMs - 1) / kNumSMs;
    const double eff = (double)ctas / (double)(waves * kNumSMs);
    if (eff > best_eff + 0.03) {
      best_eff = eff;
      best = s;
    }
  }
  while ((col_tiles + best - 1) / best > kMaxTilesPerCta) ++best;
  return best;
}

// plan_row_tiles: row tiles expected to hold anchors (<= max_row_tiles, 0 = all of them).  A caller that sizes its
// buffers for the worst case without knowing N_a on the host (the sync-free path) passes its estimate here so that
// the column splits are chosen for the CTAs that will actually run; the rest exit at once.
// local_col_tiles > 0: sweep 1 runs as two launches (local chunk, then the other chunks) with separate partial slots.
static ConPlan make_plan(long long max_row_tiles, long long max_col_tiles, long long plan_row_tiles = 0,
                         long long local_col_tiles = 0) {
  if (plan_row_tiles <= 0 || plan_row_tiles > max_row_tiles) plan_row_tiles = max_row_tiles;
  ConPlan p;
  if (local_col_tiles > 0 && local_col_tiles < max_col_tiles) {
    p.splits_local = choose_splits(plan_row_tiles, local_col_tiles);
    p.splits = choose_splits(plan_row_tiles, max_col_tiles - local_col_tiles);
  } else {
    p.splits_local = 0;
    p.splits = choose_splits(plan_row_tiles, max_col_tiles);
  }
  const int best = choose_splits(plan_row_tiles, max_col_tiles);
  p.splits2 = best > 1 ? (best + 1) / 2 : 1;
#ifdef UCD_DEBUG_KNOBS
  static const int env_s1 = getenv("UCD_SPLITS1") ? atoi(getenv("UCD_SPLITS1")) : 0;  // tuning knobs, read once
  static const int env_s2 = getenv("UCD_SPLITS2") ? atoi(getenv("UCD_SPLITS2")) : 0;
  if (env_s1 > 0) p.splits = env_s1;
  if (env_s2 > 0) p.splits2 = env_s2;
#endif
  while ((max_col_tiles + p.splits - 1) / p.splits > kMaxTilesPerCta) ++p.splits;
  while ((max_col_tiles + p.splits2 - 1) / p.splits2 > kMaxTilesPerCta) ++p.splits2;
  p.rows_pad = max_row_tiles * 128;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t r = o;
    o += (bytes + 255) & ~(size_t)255;
    return r;
  };
  p.off_stats_part = take((size_t)p.splits1_total() * 3 * p.rows_pad * 4);
  p.off_stats = take((size_t)3 * p.rows_pad * 4);
  p.off_loss_part = take((size_t)p.splits2 * 2 * p.rows_pad * 4);
  p.off_v = take((size_t)p.splits1_total() * p.rows_pad * 256 * 4);
  p.off_u = take((size_t)p.splits2 * p.rows_pad * 256 * 4);
  p.off_block = take((size_t)2 * kFinalizeBlocks * 4);
  p.total = o;
  return p;
}

template <int PHASE, int PMODE>
static int launch_sweep(const ConArgs& a, long long max_row_tiles, cudaStream_t st) {
  // the attribute is per device: set it on every call (a process may drive several GPUs), it costs ~1 us
  cudaError_t e = cudaFuncSetAttribute(con_sweep_kernel<PHASE, PMODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)kConSmem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(con_sweep_kernel)");
  const unsigned grid = (unsigned)(max_row_tiles * a.splits);
  con_sweep_kernel<PHASE, PMODE><<<grid, kConThreads, kConSmem, st>>>(a);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "con_sweep_kernel launch");
  return UCD_OK;
}

}  // namespace ucd

using namespace ucd;

extern "C" size_t ucd_con_workspace_bytes(int64_t max_row_tiles, int64_t max_col_tiles, int64_t plan_row_tiles,
                                          int64_t local_col_tiles) {
  if (max_row_tiles <= 0 || max_col_tiles <= 0) return 0;
  return make_plan(max_row_tiles, max_col_tiles, plan_row_tiles, local_col_tiles).total;
}

extern "C" int ucd_con_fwd(const void* feat_tiles, const void* prob_tiles, const int32_t* lab_tiles,
                           const int32_t* chunk_counts, int n_chunks, int64_t chunk_tiles, int64_t chunk_stride_bytes,
                           int local_chunk, int part, const void* row_feat_tiles,
                           const void* row_prob_tiles, const int32_t* row_lab_tiles, const int32_t* n_rows,
                           const int32_t* tile_range, const int32_t* row_range, int64_t self_tile0, const int32_t* min_new, int p_mode, int kpad, const float* dense_p,
                           int64_t ldp,
                           float inv_temperature, int need_grad, float* out, float* grad_unit, void* workspace,
                           size_t workspace_bytes, int64_t max_row_tiles, int64_t plan_row_tiles, void* stream) {
  UCD_CHECK_ARG(feat_tiles && lab_tiles && chunk_counts && workspace, "ucd_con_fwd: null pointer");
  UCD_CHECK_ARG(part == 1 || out, "ucd_con_fwd: null out");
  UCD_CHECK_ARG(n_chunks >= 1 && n_chunks <= kMaxChunks, "ucd_con_fwd: n_chunks=%d outside [1,%d]", n_chunks, kMaxChunks);
  UCD_CHECK_ARG(part >= 0 && part <= 2, "ucd_con_fwd: part must be 0 (all), 1 (sweep 1 over the local chunk) or 2 (the rest)");
  UCD_CHECK_ARG(part == 0 || (local_chunk >= 0 && local_chunk < n_chunks && n_chunks > 1),
                "ucd_con_fwd: a two-part run needs n_chunks > 1 and a valid local_chunk");
  UCD_CHECK_ARG(chunk_stride_bytes >= 0 && chunk_stride_bytes % 16 == 0, "ucd_con_fwd: chunk_stride_bytes must be a multiple of 16");
  UCD_CHECK_ARG(row_feat_tiles && row_lab_tiles && n_rows, "ucd_con_fwd: null row pointer");
  UCD_CHECK_ARG(tile_range && row_range, "ucd_con_fwd: null tile range pointer");
  UCD_CHECK_ARG(aligned16(row_feat_tiles) && (!row_prob_tiles || aligned16(row_prob_tiles)),
                "ucd_con_fwd: row tiles must be 16 B aligned");
  UCD_CHECK_ARG(self_tile0 >= -1 && self_tile0 < (int64_t)n_chunks * chunk_tiles, "ucd_con_fwd: bad self_tile0");
  UCD_CHECK_ARG(chunk_tiles >= 1 && max_row_tiles >= 1, "ucd_con_fwd: bad tile counts");
  UCD_CHECK_ARG(p_mode >= 0 && p_mode <= 2, "ucd_con_fwd: bad p_mode");
  UCD_CHECK_ARG(p_mode != 1 || (prob_tiles && row_prob_tiles && min_new), "ucd_con_fwd: p_mode 1 needs prob tiles and min_new");
  UCD_CHECK_ARG(p_mode != 2 || (dense_p && n_chunks == 1), "ucd_con_fwd: dense P needs a single chunk");
  UCD_CHECK_ARG(!need_grad || grad_unit || part == 1, "ucd_con_fwd: need_grad without grad_unit");
  UCD_CHECK_ARG(aligned16(feat_tiles) && aligned16(lab_tiles) && (!prob_tiles || aligned16(prob_tiles)),
                "ucd_con_fwd: tile buffers must be 16 B aligned");
  UCD_CHECK_ARG(inv_temperature > 0.f, "ucd_con_fwd: bad temperature");
  if (p_mode == 1 && (kpad < 16 || kpad > 256 || kpad % 16 != 0)) {
    set_error("ucd_con_fwd: joint-probability width kpad=%d not supported (multiple of 16 up to 256, i.e. C_old <= 256)", kpad);
    return UCD_ENOSUP;
  }
  const ConPlan plan = make_plan(max_row_tiles, (int64_t)n_chunks * chunk_tiles, plan_row_tiles, part ? chunk_tiles : 0);
  UCD_CHECK_ARG(workspace_bytes >= plan.total, "ucd_con_fwd: workspace too small (%zu < %zu)", workspace_bytes, plan.total);
  UCD_CHECK_ARG(max_row_tiles * (plan.splits > plan.splits2 ? plan.splits : plan.splits2) < (1ll << 31),
                "ucd_con_fwd: grid too large");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  ConArgs a;
  a.feat_tiles = (const __nv_bfloat16*)feat_tiles;
  a.prob_tiles = (const __nv_bfloat16*)prob_tiles;
  a.lab_tiles = lab_tiles;
  a.chunk_counts = chunk_counts;
  a.n_chunks = n_chunks;
  a.chunk_tiles = chunk_tiles;
  a.chunk_stride = chunk_stride_bytes;
  a.chunk_origin = part == 1 ? local_chunk : 0;
  a.row_feat = (const __nv_bfloat16*)row_feat_tiles;
  a.row_prob = (const __nv_bfloat16*)row_prob_tiles;
  a.row_lab = row_lab_tiles;
  a.n_rows = n_rows;
  a.tile_range = tile_range;
  a.row_range = row_range;
  a.self_tile0 = self_tile0;
  a.min_new = min_new;
  a.dense_p = dense_p;
  a.ldp = ldp;
  a.inv_tau = inv_temperature;
  a.need_grad = need_grad;
  a.kpad = kpad;
  a.rows_pad = plan.rows_pad;
  a.stats_part = (float*)(ws + plan.off_stats_part);
  a.stats = (const float*)(ws + plan.off_stats);
  a.loss_part = (float*)(ws + plan.off_loss_part);
#ifdef UCD_DEBUG_KNOBS
  a.trace = g_trace;
#else
  a.trace = nullptr;
#endif
  a.shift = 1;
  a.col_a = a.col_b = a.col_c = nullptr;
  int rc;
  // sweep 1: one launch over every chunk, or (two-part run) the local chunk first - while the exchange of the other
  // ranks' columns is still in flight - and the remaining chunks in the second call
  a.acc_part = (float*)(ws + plan.off_v);
  if (part == 1) {
    a.chunk_lo = local_chunk, a.chunk_hi = local_chunk + 1, a.chunk_skip = -1;
    a.split_base = 0, a.splits = plan.splits_local;
    return launch_sweep<1, 0>(a, max_row_tiles, st);
  }
  a.chunk_lo = 0, a.chunk_hi = n_chunks, a.chunk_skip = part == 2 ? local_chunk : -1;
  a.split_base = part == 2 ? plan.splits_local : 0, a.splits = plan.splits;
  if (part == 2) a.self_tile0 = -1;  // the anchors' own columns sit in the skipped (local) chunk
  rc = launch_sweep<1, 0>(a, max_row_tiles, st);
  if (rc != UCD_OK) return rc;
  const int splits1 = part == 2 ? plan.splits1_total() : plan.splits;
  if (a.trace) a.trace += (size_t)max_row_tiles * plan.splits * 16;  // sweep 2 counters follow sweep 1's
  con_combine_kernel<<<(unsigned)((plan.rows_pad + 255) / 256), 256, 0, st>>>(a.stats_part, splits1, plan.rows_pad,
                                                                               (float*)(ws + plan.off_stats));
  UCD_CHECK_LAUNCH("con_combine_kernel");
  // sweep 2: all chunks
  a.acc_part = (float*)(ws + plan.off_u);
  a.splits = plan.splits2;
  a.split_base = 0, a.chunk_skip = -1;
  a.self_tile0 = self_tile0;
  if (p_mode == 0)
    rc = launch_sweep<2, 0>(a, max_row_tiles, st);
  else if (p_mode == 1)
    rc = launch_sweep<2, 1>(a, max_row_tiles, st);
  else
    rc = launch_sweep<2, 2>(a, max_row_tiles, st);
  if (rc != UCD_OK) return rc;
  float* block_part = (float*)(ws + plan.off_block);
  con_finalize_kernel<<<kFinalizeBlocks, 256, 0, st>>>(a.stats, a.loss_part, (const float*)(ws + plan.off_v),
                                                       (const float*)(ws + plan.off_u), splits1, plan.splits2,
                                                       plan.rows_pad,
                                                       n_rows, inv_temperature, need_grad, grad_unit, block_part);
  UCD_CHECK_LAUNCH("con_finalize_kernel");
  con_reduce_out_kernel<<<1, 256, 0, st>>>(block_part, kFinalizeBlocks, out);
  UCD_CHECK_LAUNCH("con_reduce_out_kernel");
  return UCD_OK;
}

// ---- self-contrast losses -----------------------------------------------------------------------------------------
static size_t selfcon_extra_off(const ConPlan& p) { return (p.total + 255) & ~(size_t)255; }

extern "C" size_t ucd_selfcon_workspace_bytes(int64_t tiles) {
  if (tiles <= 0) return 0;
  const ConPlan p = make_plan(tiles, tiles);
  return selfcon_extra_off(p) + (size_t)3 * p.rows_pad * sizeof(float);
}

extern "C" int ucd_selfcon_fwd(const void* feat_tiles, const int32_t* lab_tiles, const int32_t* tile_range,
                               const int32_t* counts, const int32_t* n_rows, int64_t n, int64_t n_anchor, int mode,
                               float inv_temperature, float kappa, int need_grad, float* out, float* grad_unit,
                               void* workspace, size_t workspace_bytes, void* stream) {
  UCD_CHECK_ARG(feat_tiles && lab_tiles && tile_range && counts && n_rows && out && workspace,
                "ucd_selfcon_fwd: null pointer");
  UCD_CHECK_ARG(n >= 1 && n_anchor >= 1 && n_anchor <= n, "ucd_selfcon_fwd: bad row counts");
  UCD_CHECK_ARG(mode == 0 || mode == 1, "ucd_selfcon_fwd: mode must be 0 (PixelConLoss v1) or 1 (SupConLoss)");
  UCD_CHECK_ARG(inv_temperature > 0.f, "ucd_selfcon_fwd: bad temperature");
  UCD_CHECK_ARG(!need_grad || grad_unit, "ucd_selfcon_fwd: need_grad without grad_unit");
  UCD_CHECK_ARG(aligned16(feat_tiles) && aligned16(lab_tiles), "ucd_selfcon_fwd: tile buffers must be 16 B aligned");
  const int64_t tiles = (n + 127) / 128;
  const ConPlan plan = make_plan(tiles, tiles);
  const size_t off_x = selfcon_extra_off(plan);
  UCD_CHECK_ARG(workspace_bytes >= off_x + (size_t)3 * plan.rows_pad * sizeof(float),
                "ucd_selfcon_fwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  float* col = (float*)(ws + off_x);
  ConArgs a;
  a.feat_tiles = (const __nv_bfloat16*)feat_tiles, a.prob_tiles = nullptr, a.lab_tiles = lab_tiles;
  a.chunk_counts = counts, a.n_chunks = 1, a.chunk_tiles = tiles, a.chunk_stride = 0, a.chunk_origin = 0;
  a.chunk_lo = 0, a.chunk_hi = 1, a.chunk_skip = -1, a.split_base = 0;
  a.row_feat = (const __nv_bfloat16*)feat_tiles, a.row_prob = nullptr, a.row_lab = lab_tiles;  // rows = columns
  a.n_rows = n_rows, a.tile_range = tile_range, a.row_range = tile_range, a.self_tile0 = 0, a.min_new = nullptr;
  a.dense_p = nullptr, a.ldp = 0, a.inv_tau = inv_temperature, a.kpad = 16, a.rows_pad = plan.rows_pad;
  a.stats_part = (float*)(ws + plan.off_stats_part), a.stats = (const float*)(ws + plan.off_stats);
  a.loss_part = (float*)(ws + plan.off_loss_part), a.trace = nullptr;
  a.shift = 0;
  a.col_a = col, a.col_b = col + plan.rows_pad, a.col_c = col + 2 * plan.rows_pad;
  // sweep 1: raw row max, neg (different label), num (same label, the row itself excluded)
  a.need_grad = 0, a.splits = plan.splits, a.acc_part = (float*)(ws + plan.off_v);
  int rc = launch_sweep<1, 0>(a, tiles, st);
  if (rc != UCD_OK) return rc;
  con_combine_kernel<<<(unsigned)((plan.rows_pad + 255) / 256), 256, 0, st>>>(a.stats_part, plan.splits, plan.rows_pad,
                                                                               (float*)(ws + plan.off_stats));
  UCD_CHECK_LAUNCH("con_combine_kernel");
  // sweep 2 over the positive pairs: v1 {L_i, T_i} with the unshifted denominator, SupCon {sum s, sum exp(s)}
  a.splits = plan.splits2, a.acc_part = (float*)(ws + plan.off_u);
  rc = mode == 0 ? launch_sweep<2, 0>(a, tiles, st) : launch_sweep<2, 3>(a, tiles, st);
  if (rc != UCD_OK) return rc;
  float* block_part = (float*)(ws + plan.off_block);
  selfcon_rowcoef_kernel<<<kFinalizeBlocks, 256, 0, st>>>(a.stats, a.loss_part, plan.splits2, plan.rows_pad, n, n_anchor,
                                                          mode, inv_temperature, kappa, col, col + plan.rows_pad,
                                                          col + 2 * plan.rows_pad, block_part);
  UCD_CHECK_LAUNCH("selfcon_rowcoef_kernel");
  con_reduce_out_kernel<<<1, 256, 0, st>>>(block_part, kFinalizeBlocks, out);
  UCD_CHECK_LAUNCH("con_reduce_out_kernel");
  if (!need_grad) return UCD_OK;
  // sweep 3: H F with H = G + G^T formed pair by pair (sweep3_cols)
  a.need_grad = 1, a.splits = plan.splits, a.acc_part = (float*)(ws + plan.off_v);
  rc = mode == 0 ? launch_sweep<3, 0>(a, tiles, st) : launch_sweep<3, 1>(a, tiles, st);
  if (rc != UCD_OK) return rc;
  selfcon_grad_kernel<<<kFinalizeBlocks, 256, 0, st>>>((const float*)(ws + plan.off_v), plan.splits, plan.rows_pad, n,
                                                        inv_temperature, grad_unit);
  UCD_CHECK_LAUNCH("selfcon_grad_kernel");
  return UCD_OK;
}

extern "C" int ucd_con_bwd(const float* grad_unit, const float* out, const float* g_scalar, float g_mul,
                           const int32_t* n_rows, const int32_t* row_ref, float* d_anchor, int64_t max_rows,
                           void* stream) {
  UCD_CHECK_ARG(grad_unit && out && g_scalar && n_rows && d_anchor, "ucd_con_bwd: null pointer");
  UCD_CHECK_ARG(aligned16(grad_unit) && aligned16(d_anchor), "ucd_con_bwd: 16 B alignment required");
  if (max_rows <= 0) return UCD_OK;
  long long blocks = (max_rows * 64 + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  con_bwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(grad_unit, out, g_scalar, g_mul, n_rows, row_ref,
                                                                     d_anchor, max_rows);
  UCD_CHECK_LAUNCH("con_bwd_kernel");
  return UCD_OK;
}

#ifdef UCD_DEBUG_KNOBS
// Debug aid (not part of the product path): when set to a device buffer of
// 2 * max_row_tiles * splits * 16 int64, every CTA of the two sweeps records per-role cycle counters:
//   [0] producer total, [1] wait for a free C stage, [2] wait for the P stage, [3] tiles loaded
//   [4] MMA issuer total, [5] idle (nothing ready), [6] active tiles
//   [8] epilogue total, [9] wait for S, [10] wait for the E buffer, [11] tiles
extern "C" int ucd_con_debug_trace(void* device_buffer) {
  g_trace = (long long*)device_buffer;
  return UCD_OK;
}
extern "C" int ucd_con_debug_splits(int64_t max_row_tiles, int64_t max_col_tiles) {
  return make_plan(max_row_tiles, max_col_tiles).splits;
}
#endif  // UCD_DEBUG_KNOBS
