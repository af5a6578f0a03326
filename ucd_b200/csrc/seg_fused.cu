// N1 (SURVEY.md 8f): upsample + unbiased CE + unbiased KD fused, straight from the LOW-RES logits.
//
// Reference path being fused (train.py:108,116,133 with segmentation_module.py:133):
//   outputs     = interpolate(sem_logits    [B,C,h,w])      -> [B,C,H,W]      (grad)
//   outputs_old = interpolate(sem_logits_old[B,C_old,h,w])  -> [B,C_old,H,W]  (no grad)
//   ce = UnbiasedCrossEntropy(old_cl, 'none')(outputs, labels).mean() ; kd = UnbiasedKD(alpha)(outputs, outputs_old)
// The full-resolution logits exist only to feed these two reductions, so this kernel never writes them: every
// full-res pixel is interpolated on the fly from a low-res tile in shared memory, both losses and both
// gradients w.r.t. the full-res logits are formed in registers, and the gradients go straight through the
// adjoint of the bilinear interpolation into two small [B,C,h,w] tensors.  HBM traffic drops from
// ~(32C+12C_old+28) B per full-res pixel to the 8 B label read; the kernel is exp/issue bound.
//
// Work decomposition: block = (image b, low-res row interval k, column tile): all full-res rows Y whose upper tap
// is low-res row k (they share the y taps), TX consecutive columns, one thread per column.  For a fixed column the
// x-blend of the two tap rows, u0[c] and u1[c], is computed once per block and kept in shared memory; then
// x_c(Y) = hy0(Y) u0[c] + hy1(Y) u1[c] costs two FMAs per pixel and channel.
//   phase A (per pixel): online log-sum-exps (all / old / bkg set, old-model softmax) -> per-pixel stats in registers
//     (4 threads share a column and own every 4th row)
//   phase B (per channel, pixels of the column in the inner loop): dCE/dx_c and dKD/dx_c, accumulated over the
//     rows with the y-tap weights into 4 values per (channel, column); four channels at a time these go to shared
//     memory, and one thread per low-res cell folds the x-tap weights over the cell's (contiguous) column range and
//     the row groups in a fixed order - 3x fewer instructions than a segmented shuffle reduction per channel.
// CE-only form (KD = false, C_old = 0, no old model: the base step): phase A keeps the all-class and old-class
// log-sum-exps only, phase B forms dCE only, and shared memory, the slabs and the gather carry one gradient term.
// Cross-block sums (a low-res cell collects from <= 3 (interval, tap row) sources x <= 3 column tiles; the three loss
// sums from every block) go through per-block slabs and a second kernel that adds them in a fixed order: like the
// rest of the library the results are bit-identical from run to run (no atomics).
#include "common.cuh"

namespace ucd {

constexpr int kRG = 4;        // row groups: threads (x, g) share column x, thread g owns rows g, g+4, ...
constexpr int kRPT = 8;       // rows per thread  => up to 32 full-res rows per low-res interval (upscale <= 19)
constexpr float kNeg = -3.0e38f;

struct FusedArgs {
  const float* lr;      // [B,C,h,w]
  const float* lo;      // [B,C_old,h,w]
  long long* labels;    // [B,H,W] (remapped in place like UnbiasedCrossEntropy)
  float* g_ce;          // [B,C,h,w]  d(sum_px ce_px)/d lr
  float* g_kd;          // [B,C,h,w]  d(sum_px kd_px)/d lr, kd_px = -loss_px (unused in the CE-only form)
  float* sums;          // [3] {sum ce_px, #non-ignored, sum kd_px} (sum kd_px = 0 in the CE-only form)
  float* psum;          // workspace [3][nblk]: per-block partial sums
  float* slab;          // workspace [nblk][ncell]: per-block gradient cells (need_grad)
  int B, C, C_old, h, w, H, W, old_cl, ignore_index;
  float alpha, scale_h, scale_w;
  int need_grad;
};

// dynamic smem: u[(C + C_old)][2][TX] | abuf[kChunkC][2 NT][kRG][TX] | xw0[TX] xw1[TX] | xi0[TX] xi1[TX] | rng[ncx][4]
constexpr int kChunkC = 8;   // channels per x-reduction pass (4: 0.562 ms, 8: 0.518 ms, 16: 0.536 ms at the bench shape)
// KD: the CE + KD form; false: the CE-only form (a.C_old == 0, a.lo, a.g_kd unused).  NT gradient terms per cell.
template <int TX, bool KD>
__global__ void __launch_bounds__(TX * kRG) seg_fused_kernel(const FusedArgs a, int ncx_cap) {
  extern __shared__ __align__(16) float fs[];
  constexpr int NW = TX * kRG / 32;
  constexpr int NT = KD ? 2 : 1;
  const int C = a.C, Co = KD ? a.C_old : 0, CT = C + Co;
  float* u = fs;                               // [CT][2][TX]  x-blended tap rows per column
  // [kChunkC * 2 NT planes][kRG][TX] y-reduced gradient terms of one channel chunk; the plane stride is odd so that
  // the 16 planes a warp of the x pass reads at the same (row group, column) fall into different banks
  constexpr int PS = kRG * TX + 1;
  float* abuf = u + (size_t)CT * 2 * TX;
  float* xw0 = abuf + kChunkC * 2 * NT * PS + 3;  // x-tap weights of the tile's columns
  float* xw1 = xw0 + TX;
  int* xi0 = reinterpret_cast<int*>(xw1 + TX);  // tile-local low-res column of each tap (-1: column outside the image)
  int* xi1 = xi0 + TX;
  int* rng = xi1 + TX;                          // [ncx_cap][4]: column ranges [a0,b0) with i0 == cell, [a1,b1) with i1 == cell
  __shared__ float red[3][NW];

  const int b = blockIdx.z, k = blockIdx.y, X0 = blockIdx.x * TX;
  const int xl = threadIdx.x % TX, rg = threadIdx.x / TX;
  const int X = X0 + xl;
  const bool colok = X < a.W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // rows of this interval: all Y with tap.i0 == k (contiguous).  Found by scanning a conservative range.
  int Ya = a.H, Yb = -1;
  {
    const float inv = (float)a.H / (float)a.h;
    int lo_ = (int)floorf(((float)k - 0.5f) * inv) - 2, hi_ = (int)ceilf(((float)k + 1.5f) * inv) + 2;
    lo_ = max(lo_, 0), hi_ = min(hi_, a.H - 1);
    if (a.h == a.H) lo_ = hi_ = k;
    for (int Y = lo_; Y <= hi_; ++Y) {
      if (bilinear_tap(Y, a.scale_h, a.h, a.H).i0 == k) {
        Ya = min(Ya, Y);
        Yb = max(Yb, Y);
      }
    }
  }
  const int nrow = Yb - Ya + 1;
  const int blk = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
  const int nblk = gridDim.x * gridDim.y * gridDim.z;
  const int ncell = 2 * ncx_cap * C * NT;
  if (nrow <= 0) {  // uniform per block (cannot happen when upsampling; kept for safety): contributes zeros
    if (threadIdx.x < 3) a.psum[(size_t)threadIdx.x * nblk + blk] = 0.f;
    if (a.need_grad)
      for (int i = threadIdx.x; i < ncell; i += TX * kRG) a.slab[(size_t)blk * ncell + i] = 0.f;
    return;
  }
  const int k1 = min(k + 1, a.h - 1);  // lower tap row (weight 0 when clamped)

  const Tap tx = bilinear_tap(colok ? X : a.W - 1, a.scale_w, a.w, a.W);
  // the labels of this thread's rows come from HBM: request them now, they arrive while the tap rows are staged
  long long lab_pre[kRPT];
#pragma unroll
  for (int j = 0; j < kRPT; ++j) {
    const int r = rg + j * kRG;
    lab_pre[j] = (r < nrow && colok) ? a.labels[((size_t)b * a.H + Ya + r) * a.W + X] : 0;
  }
  // x-blended tap rows for every channel of this column (channels split over the row groups)
  {
    const float* pn = a.lr + (size_t)b * C * a.h * a.w;
    const float* po = KD ? a.lo + (size_t)b * Co * a.h * a.w : nullptr;
    for (int c = rg; c < CT; c += kRG) {
      const float* p = (c < C) ? pn + (size_t)c * a.h * a.w : po + (size_t)(c - C) * a.h * a.w;
      const float v00 = __ldg(p + k * a.w + tx.i0), v01 = __ldg(p + k * a.w + tx.i1);
      const float v10 = __ldg(p + k1 * a.w + tx.i0), v11 = __ldg(p + k1 * a.w + tx.i1);
      // ATen's generic kernel order: t = fma(v0, w0, v1*w1), out = fma(t0, h0, t1*h1)
      u[((size_t)c * 2 + 0) * TX + xl] = __fmaf_rn(v00, tx.w0, __fmul_rn(v01, tx.w1));
      u[((size_t)c * 2 + 1) * TX + xl] = __fmaf_rn(v10, tx.w0, __fmul_rn(v11, tx.w1));
    }
  }
  __syncthreads();

  const float a2 = a.alpha * kLog2e;
  const float inv_co = 1.f / (float)Co;
  float ce_acc = 0.f, valid_acc = 0.f, kd_acc = 0.f;
  // per-pixel statistics of this thread's rows (registers)
  float s_lse2[kRPT], s_fold[kRPT], s_fb[kRPT], s_lt2[kRPT], s_h0[kRPT], s_h1[kRPT];
  int s_lab[kRPT];
  // ---------------- phase A: channels in the outer loop, 4 rows of the thread in flight (independent chains) ----
#pragma unroll
  for (int j = 0; j < kRPT; ++j) {
    s_lab[j] = -1;
    s_lse2[j] = 0.f, s_fold[j] = 0.f, s_fb[j] = 0.f, s_lt2[j] = 0.f, s_h0[j] = 0.f, s_h1[j] = 0.f;
  }
#pragma unroll
  for (int jb = 0; jb < kRPT; jb += 4) {
    if (rg + jb * kRG >= nrow) break;
    long long lab[4];
    float h0[4], h1[4];
    bool live[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int r = rg + (jb + q) * kRG;
      live[q] = r < nrow;
      const int Y = Ya + (live[q] ? r : 0);
      const Tap ty = bilinear_tap(Y, a.scale_h, a.h, a.H);
      h0[q] = ty.w0, h1[q] = ty.w1;
      lab[q] = 0;
      if (live[q] && colok) {
        long long* lp = a.labels + ((size_t)b * a.H + Y) * a.W + X;
        lab[q] = lab_pre[jb + q];
        if (lab[q] < a.old_cl) {  // utils/loss.py:104-105
          if (lab[q] != 0) *lp = 0;
          lab[q] = 0;
        }
      }
    }
    float m[4], s[4], mo[4], so[4], mb[4], sb[4], picked[4], mt[4], stt[4], wx[4], t0v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      m[q] = mo[q] = mb[q] = mt[q] = kNeg, s[q] = so[q] = sb[q] = stt[q] = 0.f, picked[q] = wx[q] = t0v[q] = 0.f;
    for (int c = 0; c < C; ++c) {
      const float u0 = u[((size_t)c * 2) * TX + xl], u1 = u[((size_t)c * 2 + 1) * TX + xl];
      const bool bkg = (c == 0 || c >= Co);
      float v0 = 0.f, v1 = 0.f;
      if (c < Co) v0 = u[((size_t)(C + c) * 2) * TX + xl], v1 = u[((size_t)(C + c) * 2 + 1) * TX + xl];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float x = __fmaf_rn(u0, h0[q], __fmul_rn(u1, h1[q]));
        const float x2 = x * kLog2e;
        if (c == a.old_cl) mo[q] = m[q], so[q] = s[q];  // snapshot: log-sum-exp over the first old_cl channels
        lse_push(m[q], s[q], x2);
        if (KD && bkg) lse_push(mb[q], sb[q], x2);
        picked[q] = (lab[q] == c) ? x : picked[q];
        if (KD && c < Co) {
          const float tv = __fmaf_rn(v0, h0[q], __fmul_rn(v1, h1[q])) * a2;
          if (c == 0) t0v[q] = tv;
          const float d = tv - mt[q];
          const float e = ex2f(-fabsf(d));
          const float xc = c >= 1 ? x : 0.f;
          stt[q] = d > 0.f ? fmaf(stt[q], e, 1.f) : stt[q] + e;
          wx[q] = d > 0.f ? fmaf(wx[q], e, xc) : fmaf(e, xc, wx[q]);
          mt[q] = fmaxf(mt[q], tv);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = jb + q;
      if (!live[q]) continue;
      if (a.old_cl >= C) mo[q] = m[q], so[q] = s[q];
      const float lse2 = m[q] + lg2f(s[q]), lseo2 = mo[q] + lg2f(so[q]), lseb2 = mb[q] + lg2f(sb[q]);
      const float lset2 = mt[q] + lg2f(stt[q]);
      const float lse = lse2 * kLn2;
      const bool ign = lab[q] == a.ignore_index;
      const bool dead = ign || lab[q] < 0 || lab[q] >= C;
      float l = (lab[q] == 0 && a.old_cl > 0) ? (lse - lseo2 * kLn2) : (lse - picked[q]);
      if (dead) l = 0.f;
      const float q0 = ex2f(t0v[q] - lset2);
      const float kdpx = -((q0 * (lseb2 * kLn2 - lse) + wx[q] / stt[q] - (1.f - q0) * lse) * inv_co);
      if (colok) {
        ce_acc += l;
        valid_acc += ign ? 0.f : 1.f;
        if (KD) kd_acc += kdpx;
      }
      // phase B sees: label -1 = no CE gradient (ignored / out of image), -2 = background-remapped pixel (its CE
      // gradient subtracts p_c exp(lse - lse_old) over the old classes; s_fold is 0 for every other pixel)
      const bool off = dead || !colok;
      const bool isbkg = !off && lab[q] == 0 && a.old_cl > 0;
      s_lse2[j] = lse2;
      s_fold[j] = isbkg ? ex2f(lse2 - lseo2) : 0.f;  // exp(lse - lse_old)
      s_fb[j] = q0 * ex2f(lse2 - lseb2);             // q0 exp(lse - lse_bkg)
      s_lt2[j] = lset2;
      s_lab[j] = off ? -1 : (isbkg ? -2 : (int)lab[q]);
      s_h0[j] = colok ? h0[q] : 0.f;        // out-of-image columns contribute nothing
      s_h1[j] = colok ? h1[q] : 0.f;
    }
  }
  {
    float v0 = warp_sum(ce_acc), v1 = warp_sum(valid_acc), v2 = warp_sum(kd_acc);
    if (lane == 0) red[0][warp] = v0, red[1][warp] = v1, red[2][warp] = v2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int i = 0; i < NW; ++i) s0 += red[0][i], s1 += red[1][i], s2 += red[2][i];
    a.psum[blk] = s0;
    a.psum[(size_t)nblk + blk] = s1;
    a.psum[2 * (size_t)nblk + blk] = s2;
  }
  if (!a.need_grad) return;

  // ---------------- phase B: gradients, one channel at a time ----------------
  const int cx_lo = bilinear_tap(min(X0, a.W - 1), a.scale_w, a.w, a.W).i0;  // first low-res column of this tile
  const int nj = (nrow + kRG - 1) / kRG;  // rows per thread that exist in this interval
  // x-tap tables of the tile and, per low-res cell, the contiguous ranges of columns whose taps hit it
  for (int i = threadIdx.x; i < ncx_cap * 4; i += TX * kRG) rng[i] = 0;
  if (rg == 0) {
    xw0[xl] = tx.w0, xw1[xl] = tx.w1;
    xi0[xl] = colok ? tx.i0 - cx_lo : -1;
    xi1[xl] = colok ? tx.i1 - cx_lo : -1;
  }
  __syncthreads();
  if (rg == 0 && colok) {
    const int i0 = xi0[xl], i1 = xi1[xl];
    if (xl == 0 || xi0[xl - 1] != i0) rng[i0 * 4 + 0] = xl;
    if (xl == TX - 1 || xi0[xl + 1] != i0) rng[i0 * 4 + 1] = xl + 1;
    if (xl == 0 || xi1[xl - 1] != i1) rng[i1 * 4 + 2] = xl;
    if (xl == TX - 1 || xi1[xl + 1] != i1) rng[i1 * 4 + 3] = xl + 1;
  }
  // (the first pass below is preceded by a __syncthreads)
  for (int c = 0; c < C; ++c) {
    const float u0 = u[((size_t)c * 2) * TX + xl], u1 = u[((size_t)c * 2 + 1) * TX + xl];
    float v0 = 0.f, v1 = 0.f;
    if (KD && c < Co) v0 = u[((size_t)(C + c) * 2) * TX + xl], v1 = u[((size_t)(C + c) * 2 + 1) * TX + xl];
    const bool in_sb = (c == 0) || (c >= Co);
    const bool old_fg = (c >= 1) && (c < Co);
    const float oldc = (c < a.old_cl) ? 1.f : 0.f;  // uniform: channel c belongs to the old classes
    float ce0 = 0.f, ce1 = 0.f, kd0 = 0.f, kd1 = 0.f;
#pragma unroll
    for (int j = 0; j < kRPT; ++j) {
      if (j >= nj) break;  // block-uniform: an interior 16x interval has 16 rows = 4 per thread, not kRPT
      const float h0 = s_h0[j], h1 = s_h1[j];  // zero for rows this thread does not own
      const float x = __fmaf_rn(u0, h0, __fmul_rn(u1, h1));
      const int lab = s_lab[j];
      const float p = ex2f(fmaf(x, kLog2e, -s_lse2[j]));
      // dCE/dx_c = p_c - [old c] p_c fold - [c == label]   (fold = 0 unless the pixel was remapped to background)
      const float sub = fmaf(p * oldc, s_fold[j], (c == lab) ? 1.f : 0.f);
      const float dce = (lab == -1) ? 0.f : (p - sub);
      ce0 = fmaf(h0, dce, ce0);
      ce1 = fmaf(h1, dce, ce1);
      if (KD) {
        float dkd = p;
        if (in_sb) dkd -= p * s_fb[j];
        if (old_fg) dkd -= ex2f(fmaf(__fmaf_rn(v0, h0, __fmul_rn(v1, h1)), a2, -s_lt2[j]));
        dkd *= inv_co;
        kd0 = fmaf(h0, dkd, kd0);
        kd1 = fmaf(h1, dkd, kd1);
      }
    }
    // park the four y-reduced terms of this channel; every kChunkC channels one thread per cell folds the x taps
    {
      const int cl = c % kChunkC;
      float* ab = abuf + (size_t)cl * 2 * NT * PS + rg * TX + xl;
      ab[0] = ce0, ab[PS] = ce1;
      if (KD) ab[2 * PS] = kd0, ab[3 * PS] = kd1;
    }
    if ((c + 1) % kChunkC == 0 || c == C - 1) {
      const int c_first = c - (c % kChunkC);
      __syncthreads();
      // work item = (output cell value, tap side): adjacent lanes take the i0 / i1 column range of one output and
      // exchange their partial sums; four row-group chains per thread keep the FMA pipe busy
      const int n_out = 2 * ncx_cap * kChunkC * NT;  // (yy, cx, channel of the chunk, term)
      for (int w2 = threadIdx.x; w2 < ((2 * n_out + 31) & ~31); w2 += TX * kRG) {
        const int side = w2 & 1, o = w2 >> 1;
        const bool live = o < n_out;
        const int term = KD ? o & 1 : 0, cl = (o >> (NT - 1)) % kChunkC;
        const int cx = live ? (o / (NT * kChunkC)) % ncx_cap : 0, yy = live ? (o / (NT * kChunkC)) / ncx_cap : 0;
        const int cc = c_first + cl;
        const float* ab = abuf + ((size_t)cl * 2 * NT + (term * 2 + yy)) * PS;
        const float* xw = side ? xw1 : xw0;
        const int xa = live ? rng[cx * 4 + 2 * side] : 0, xb = live ? rng[cx * 4 + 2 * side + 1] : 0;
        float acc[kRG];
#pragma unroll
        for (int g = 0; g < kRG; ++g) acc[g] = 0.f;
#pragma unroll 4
        for (int x = xa; x < xb; ++x) {
          const float wv = xw[x];
#pragma unroll
          for (int g = 0; g < kRG; ++g) acc[g] = fmaf(wv, ab[(size_t)g * TX + x], acc[g]);
        }
        const float mine = (acc[0] + acc[1]) + (acc[2] + acc[3]);  // fixed order: deterministic
        const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
        if (live && side == 0 && cc <= c)
          a.slab[(size_t)blk * ncell + (((size_t)yy * ncx_cap + cx) * C + cc) * NT + term] = mine + other;
      }
      __syncthreads();
    }
  }
}

// Second stage: fixed-order sums of the per-block slabs.  One thread per low-res element (b, c, gy, gx), both terms.
// Sources of row gy: interval gy as its upper tap row (yy = 0), interval gy-1 as its lower tap row (yy = 1), and - at
// the bottom border, where the lower tap is clamped - interval h-1's lower tap row again.  KD = false: dCE only.
template <bool KD>
__global__ void __launch_bounds__(256)
seg_fused_gather_kernel(const FusedArgs a, int TX, int ntx, int ncx_cap) {
  constexpr int NT = KD ? 2 : 1;
  const int C = a.C;
  const size_t ncell = (size_t)2 * ncx_cap * C * NT;
  const long long n = (long long)a.B * C * a.h * a.w;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int gx = (int)(i % a.w), gy = (int)((i / a.w) % a.h);
    const int c = (int)((i / ((long long)a.w * a.h)) % C), b = (int)(i / ((long long)a.w * a.h * C));
    float ce = 0.f, kd = 0.f;
    for (int src = 0; src < 3; ++src) {
      int k, yy;
      if (src == 0) k = gy, yy = 0;
      else if (src == 1) k = gy - 1, yy = 1;
      else k = a.h - 1, yy = 1;
      if (k < 0 || (src == 2 && gy != a.h - 1)) continue;
      for (int t = 0; t < ntx; ++t) {
        const int cx = gx - bilinear_tap(min(t * TX, a.W - 1), a.scale_w, a.w, a.W).i0;
        if (cx < 0 || cx >= ncx_cap) continue;
        const size_t blk = ((size_t)b * a.h + k) * ntx + t;
        if (KD) {
          const float2 v = *reinterpret_cast<const float2*>(a.slab + blk * ncell + (((size_t)yy * ncx_cap + cx) * C + c) * 2);
          ce += v.x, kd += v.y;
        } else {
          ce += a.slab[blk * ncell + ((size_t)yy * ncx_cap + cx) * C + c];
        }
      }
    }
    a.g_ce[i] = ce;
    if (KD) a.g_kd[i] = kd;
  }
}

__global__ void __launch_bounds__(1024)
seg_fused_sums_kernel(const float* __restrict__ psum, int nblk, float* __restrict__ sums) {
  __shared__ float red[32];
  const int k = blockIdx.x;  // one block per sum, fixed order
  float acc = 0.f;
  for (int i = threadIdx.x; i < nblk; i += blockDim.x) acc += psum[(size_t)k * nblk + i];
  const float r = block_sum(acc, red);
  if (threadIdx.x == 0) sums[k] = r;
}

struct FusedPlan {
  int TX, ncx, ntx;
  size_t smem;
  long long nblk;
  size_t ncell, floats;  // workspace: psum [3][nblk] (padded to 4 floats) then slab [nblk][ncell]
};

// C_old == 0 plans the CE-only form: one gradient term per cell instead of two
static bool fused_plan(int B, int C, int C_old, int h, int w, int W, FusedPlan& p) {
  // column tile: the widest of {128, 64, 32} whose shared memory fits
  const int CT = C + C_old, NT = C_old > 0 ? 2 : 1;
  p.TX = 0;
  for (int cand : {128, 64, 32}) {
    const int ncx = (int)((double)cand * w / W) + 3;
    const size_t need = ((size_t)CT * 2 * cand + (size_t)kChunkC * 2 * NT * (kRG * cand + 1) + 3 + 4 * (size_t)cand +
                         4 * (size_t)ncx) * sizeof(float);
    if (need <= 72 * 1024 || (cand == 32 && need <= 200 * 1024)) {  // prefer >= 3 blocks per SM
      p.TX = cand, p.smem = need, p.ncx = ncx;
      break;
    }
  }
  if (p.TX == 0) return false;
  p.ntx = (W + p.TX - 1) / p.TX;
  p.nblk = (long long)B * h * p.ntx;
  p.ncell = (size_t)2 * p.ncx * C * NT;
  p.floats = (((size_t)3 * p.nblk + 3) & ~(size_t)3) + (size_t)p.nblk * p.ncell;
  return true;
}

}  // namespace ucd

using namespace ucd;

extern "C" size_t ucd_seg_fused_workspace_floats(int B, int C, int C_old, int h, int w, int H, int W) {
  (void)H;
  FusedPlan p;
  if (B <= 0 || C <= 0 || C_old < 0 || h <= 0 || w <= 0 || W < w || !fused_plan(B, C, C_old, h, w, W, p)) return 0;
  return p.floats;
}

extern "C" int ucd_seg_fused_fwd(const float* lr, const float* lr_old, int64_t* labels, float* g_ce, float* g_kd,
                                 float* sums, float* workspace, size_t workspace_floats, int B, int C, int C_old, int h,
                                 int w, int H, int W, int old_cl, int ignore_index, float alpha, int need_grad,
                                 void* stream) {
  const bool kd = C_old > 0;  // C_old == 0: the CE-only form (no old model; lr_old and g_kd are not read)
  UCD_CHECK_ARG(lr && (lr_old || !kd) && labels && sums && workspace, "ucd_seg_fused_fwd: null pointer");
  UCD_CHECK_ARG(!need_grad || (g_ce && (g_kd || !kd)), "ucd_seg_fused_fwd: need_grad without gradient buffers");
  UCD_CHECK_ARG(B > 0 && C > 0 && C_old >= 0 && C >= C_old && h > 0 && w > 0 && H >= h && W >= w,
                "ucd_seg_fused_fwd: bad shape (upsampling only)");
  UCD_CHECK_ARG(old_cl >= 0 && old_cl <= C, "ucd_seg_fused_fwd: old_cl outside [0,C]");
  UCD_CHECK_ARG(B <= 65535 && h <= 65535, "ucd_seg_fused_fwd: batch / rows too large for the grid");
  UCD_CHECK_ARG(aligned16(workspace), "ucd_seg_fused_fwd: workspace must be 16 B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int rows_cap = (int)(1.5 * (double)H / h) + 3;  // the first interval also owns the clamped rows above row 0
  UCD_CHECK_ARG(rows_cap <= kRG * kRPT, "ucd_seg_fused_fwd: upscale factor %d too large for the fused kernel (max 19)", H / h);
  FusedPlan p;
  UCD_CHECK_ARG(fused_plan(B, C, C_old, h, w, W, p), "ucd_seg_fused_fwd: C + C_old = %d too large for one block", C + C_old);
  UCD_CHECK_ARG(workspace_floats >= p.floats, "ucd_seg_fused_fwd: workspace too small (%zu < %zu floats)",
                workspace_floats, p.floats);
  UCD_CHECK_ARG(p.nblk < (1ll << 31), "ucd_seg_fused_fwd: too many blocks");
  FusedArgs a;
  a.lr = lr, a.lo = lr_old, a.labels = (long long*)labels, a.g_ce = g_ce, a.g_kd = g_kd, a.sums = sums;
  a.psum = workspace, a.slab = workspace + (((size_t)3 * p.nblk + 3) & ~(size_t)3);
  a.B = B, a.C = C, a.C_old = C_old, a.h = h, a.w = w, a.H = H, a.W = W, a.old_cl = old_cl, a.ignore_index = ignore_index;
  a.alpha = alpha, a.scale_h = (float)h / (float)H, a.scale_w = (float)w / (float)W, a.need_grad = need_grad;
  const int TX = p.TX, ncx = p.ncx;
  const size_t smem = p.smem;
  cudaError_t e;
  dim3 grid(p.ntx, h, B);
#define UCD_LAUNCH_FUSED(T, K)                                                                                       \
  do {                                                                                                               \
    if (smem > 48 * 1024) {                                                                                          \
      e = cudaFuncSetAttribute(seg_fused_kernel<T, K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);      \
      if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(seg_fused_kernel)");                           \
    }                                                                                                                \
    seg_fused_kernel<T, K><<<grid, T * kRG, smem, st>>>(a, ncx);                                                     \
  } while (0)
  if (kd) {
    if (TX == 128)
      UCD_LAUNCH_FUSED(128, true);
    else if (TX == 64)
      UCD_LAUNCH_FUSED(64, true);
    else
      UCD_LAUNCH_FUSED(32, true);
  } else {
    if (TX == 128)
      UCD_LAUNCH_FUSED(128, false);
    else if (TX == 64)
      UCD_LAUNCH_FUSED(64, false);
    else
      UCD_LAUNCH_FUSED(32, false);
  }
#undef UCD_LAUNCH_FUSED
  UCD_CHECK_LAUNCH("seg_fused_kernel");
  seg_fused_sums_kernel<<<3, 1024, 0, st>>>(a.psum, (int)p.nblk, sums);
  UCD_CHECK_LAUNCH("seg_fused_sums_kernel");
  if (need_grad) {
    const long long n = (long long)B * C * h * w;
    long long blocks = (n + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    if (kd)
      seg_fused_gather_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(a, TX, p.ntx, ncx);
    else
      seg_fused_gather_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(a, TX, p.ntx, ncx);
    UCD_CHECK_LAUNCH("seg_fused_gather_kernel");
  }
  return UCD_OK;
}
