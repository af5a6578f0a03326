// Tap tables of the sweep-form bilinear adjoint (integer upscale factors that are a multiple of 8 along x): shared by
// upsample_bwd_sweep_kernel (upsample.cu) and the UNCE + UNKD backward that folds the adjoint in (ce_kd.cu).
// One block row = W / 4 threads; thread `tid` owns the 4 consecutive full-res X = 4 tid, which share one pair of
// x taps.
#pragma once
#include "common.cuh"

namespace ucd {

// x side.  wx0 / wx1: the thread's x weights towards its upper / lower x tap; s_x0 / s_x1 [wv] scratch; s_j [w]: the
// contiguous thread ranges [x, y) whose upper tap and [z, w) whose lower tap hit each low-res column (taps are
// monotone in X).  Ends with the table written by threads < w (the caller's next barrier publishes it).
__device__ __forceinline__ void sweep_x_taps(int tid, int wv, int w, int W, float scale_w, float (&wx0)[4],
                                             float (&wx1)[4], int* s_x0, int* s_x1, short4* s_j) {
  const int X = tid * 4;
  {
    const Tap t0 = bilinear_tap(X, scale_w, w, W);
    s_x0[tid] = t0.i0, s_x1[tid] = t0.i1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const Tap tx = bilinear_tap(X + i, scale_w, w, W);  // same i0 / i1 as t0 (host-checked precondition)
      wx0[i] = tx.w0, wx1[i] = tx.w1;
    }
  }
  __syncthreads();
  if (tid < w) {
    const int sc4 = (W / w) / 4;
    const int j0 = max((tid - 2) * sc4 - 2, 0), j1 = min((tid + 2) * sc4 + 2, wv - 1);
    int a0 = 0, a1 = 0, b0 = 0, b1 = 0;
    bool fa = false, fb = false;
    for (int j = j0; j <= j1; ++j) {
      if (s_x0[j] == tid) {
        if (!fa) a0 = j, fa = true;
        a1 = j + 1;
      }
      if (s_x1[j] == tid) {
        if (!fb) b0 = j, fb = true;
        b1 = j + 1;
      }
    }
    s_j[tid] = make_short4((short)a0, (short)a1, (short)b0, (short)b1);
  }
}

// y side, for the low-res rows [y0, ylast] of one plane: s_k[i] / s_h[i] = upper-tap row and (upper, lower) y weights
// of full-res row Ylo + i (bottom border: both taps on one row, folded into the upper weight).  Returns Ylo; [i_lo,
// i_hi) are the rows whose upper tap lies in [y0, ylast] - the ones to read (the rest of the conservative range are
// margins; s_k is monotone, so exactly one row starts and one row ends that run).
__device__ __forceinline__ int sweep_y_taps(int tid, int nthr, int y0, int ylast, int h, int H, float scale_h, int ny_cap,
                                            int* s_k, float2* s_h, int* s_lim, int& i_lo, int& i_hi) {
  const float inv = (float)H / (float)h;
  int Ylo = (int)floorf(((float)y0 - 0.5f) * inv) - 2, Yhi = (int)ceilf(((float)ylast + 1.5f) * inv) + 2;
  Ylo = max(Ylo, 0), Yhi = min(Yhi, H - 1);
  const int ny = min(Yhi - Ylo + 1, ny_cap);
  __syncthreads();  // a previous segment no longer reads the tap table
  for (int i = tid; i < ny; i += nthr) {
    const Tap ty = bilinear_tap(Ylo + i, scale_h, h, H);
    s_k[i] = ty.i0;
    const bool clamped = ty.i1 == ty.i0;
    s_h[i] = make_float2(clamped ? ty.w0 + ty.w1 : ty.w0, clamped ? 0.f : ty.w1);
  }
  __syncthreads();
  for (int i = tid; i < ny; i += nthr) {
    const int k = s_k[i];
    if (k >= y0 && k <= ylast) {
      if (i == 0 || s_k[i - 1] < y0) s_lim[0] = i;
      if (i == ny - 1 || s_k[i + 1] > ylast) s_lim[1] = i + 1;
    }
  }
  __syncthreads();
  i_lo = s_lim[0], i_hi = s_lim[1];
  return Ylo;
}

}  // namespace ucd
