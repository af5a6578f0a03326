// Bilinear logit upsample (align_corners=False) and its adjoint.
// Reference: segmentation_module.py:133  F.interpolate(sem_logits, size=out_size, mode="bilinear").
//
// Forward is write-bound (4 B per output element; every low-res value is reused ~(H/h)*(W/w) times
// and stays in L1/L2): a thread owns 4 consecutive output x of one output row and loops over the
// planes of its image block, so tap indices/weights are computed once and every store is a
// coalesced 128-bit streaming store.
// Backward is read-bound (4 B per full-res gradient element): a block owns RY low-res rows of one
// plane, streams the full-res rows that touch them once (coalesced), reduces them along y in
// registers, then along x out of shared memory.  No atomics; summation order is fixed.
#include "common.cuh"
#include "sweep_adjoint.cuh"

#include <stdlib.h>

namespace ucd {

constexpr int kUpThreads = 256;

// Forward.  A thread owns VEC consecutive output x of one output row and loops over the planes of its
// plane group.  blockIdx.x covers (Y, X/VEC) flattened, blockIdx.y the plane group.
template <int VEC>
__global__ void __launch_bounds__(kUpThreads)
upsample_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, long long planes, int h, int w, int H,
                    int W, float scale_h, float scale_w, int planes_per_block) {
  const int wv = (W + VEC - 1) / VEC;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)H * wv) return;
  const int Y = (int)(idx / wv);
  const int X = (int)(idx - (long long)Y * wv) * VEC;
  const Tap ty = bilinear_tap(Y, scale_h, h, H);
  int x0[VEC], x1[VEC];
  float wx0[VEC], wx1[VEC];
  const bool small_out = H + W <= 128;  // selects ATen's operation order (bit-exact parity with the CPU reference)
  bool uniform = true;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const Tap tx = bilinear_tap(X + i, scale_w, w, W);
    x0[i] = tx.i0, x1[i] = tx.i1, wx0[i] = tx.w0, wx1[i] = tx.w1;
    uniform = uniform && tx.i0 == x0[0] && tx.i1 == x1[0];
  }
  const long long p0 = (long long)blockIdx.y * planes_per_block;
  const long long p1 = (p0 + planes_per_block < planes) ? p0 + planes_per_block : planes;
  const size_t in_plane = (size_t)h * w, out_plane = (size_t)H * W;
  float* dst = out + p0 * out_plane + (size_t)Y * W + X;
  if (uniform) {
    // All VEC outputs read the same 2x2 source cell (always the case for upscale factors that are a multiple of
    // 2*VEC, e.g. the 16x of DeepLab): 4 loads per plane, UP planes in flight.
    const float* s00 = in + p0 * in_plane + ty.i0 * w + x0[0];
    const int d01 = x1[0] - x0[0], d10 = (ty.i1 - ty.i0) * w;
    constexpr int UP = 4;
    long long p = p0;
    for (; p + UP <= p1; p += UP) {
      float v[UP][4];
#pragma unroll
      for (int u = 0; u < UP; ++u) {
        const float* s = s00 + u * in_plane;
        v[u][0] = __ldg(s), v[u][1] = __ldg(s + d01), v[u][2] = __ldg(s + d10), v[u][3] = __ldg(s + d10 + d01);
      }
#pragma unroll
      for (int u = 0; u < UP; ++u) {
        float r[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i)
          r[i] = bilinear_blend(small_out, v[u][0], v[u][1], v[u][2], v[u][3], ty.w0, ty.w1, wx0[i], wx1[i]);
        if (VEC == 4)  // streaming (evict-first) stores: 5.1 TB/s vs 3.3 TB/s with default stores (scripts/up_probe.py)
          stg_stream4(dst + u * out_plane, make_float4(r[0], r[1], r[2], r[3]));
        else
          stg_stream1(dst + u * out_plane, r[0]);
      }
      s00 += UP * in_plane;
      dst += UP * out_plane;
    }
    for (; p < p1; ++p) {
      const float a = __ldg(s00), b = __ldg(s00 + d01), c = __ldg(s00 + d10), d = __ldg(s00 + d10 + d01);
      float r[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) r[i] = bilinear_blend(small_out, a, b, c, d, ty.w0, ty.w1, wx0[i], wx1[i]);
      if (VEC == 4)
        stg_stream4(dst, make_float4(r[0], r[1], r[2], r[3]));
      else
        stg_stream1(dst, r[0]);
      s00 += in_plane;
      dst += out_plane;
    }
    return;
  }
  for (long long p = p0; p < p1; ++p) {
    const float* src = in + p * in_plane;
    float r[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i)
      r[i] = bilinear_blend(small_out, __ldg(src + ty.i0 * w + x0[i]), __ldg(src + ty.i0 * w + x1[i]),
                            __ldg(src + ty.i1 * w + x0[i]), __ldg(src + ty.i1 * w + x1[i]), ty.w0, ty.w1, wx0[i],
                            wx1[i]);
    if (VEC == 4)
      stg_stream4(dst, make_float4(r[0], r[1], r[2], r[3]));
    else
      stg_stream1(dst, r[0]);
    dst += out_plane;
  }
}

// Forward, interval form (the one the training shapes take).  block = (plane, low-res row interval k, column tile):
// all output rows whose upper tap is source row k are contiguous in memory and share both source rows, so
//   out(Y, X) = fma(t0(X), h0(Y), t1(X) * h1(Y))   with  t_r(X) = fma(v_r0, w0, v_r1 * w1)
// (exactly ATen's generic-kernel operation order) costs one FMUL + one FMA per output after 4 loads per thread.
// Consecutive blocks write consecutive ~32 KB runs: the whole grid is one sequential write stream.
constexpr int kUpMaxIvRows = 96;  // candidate rows of one interval (2*scale + 5): scale factors up to 40
template <int VEC>
__global__ void __launch_bounds__(kUpThreads)
upsample_fwd_interval_kernel(const float* __restrict__ in, float* __restrict__ out, int h, int w, int H, int W,
                             float scale_h, float scale_w, int tw, int n_col_tiles) {
  __shared__ float s_h0[kUpMaxIvRows], s_h1[kUpMaxIvRows];
  __shared__ int s_lo[3], s_hi[3];
  const int wv = (W + VEC - 1) / VEC;
  const int rp = kUpThreads / tw;  // rows per pass
  const int per_plane = h * n_col_tiles;
  const long long plane = blockIdx.x / per_plane;
  const int rem = (int)(blockIdx.x - plane * per_plane);
  const int k = rem / n_col_tiles, col_tile = rem - k * n_col_tiles;
  // rows of this interval: all Y with tap.i0 == k (contiguous); candidates evaluated in parallel by 3 warps
  const float inv = (float)H / (float)h;
  int lo = (int)floorf(((float)k - 0.5f) * inv) - 2, hi = (int)ceilf(((float)k + 1.5f) * inv) + 2;
  lo = max(lo, 0), hi = min(hi, H - 1);
  if (threadIdx.x < kUpMaxIvRows) {
    const int Y = lo + (int)threadIdx.x;
    bool match = false;
    if (Y <= hi) {
      const Tap ty = bilinear_tap(Y, scale_h, h, H);
      match = ty.i0 == k;
      s_h0[threadIdx.x] = ty.w0, s_h1[threadIdx.x] = ty.w1;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, match);
    if ((threadIdx.x & 31) == 0) {
      const int wq = threadIdx.x >> 5;
      s_lo[wq] = bal ? wq * 32 + __ffs(bal) - 1 : 1 << 30;
      s_hi[wq] = bal ? wq * 32 + 31 - __clz(bal) : -1;
    }
  }
  __syncthreads();
  const int ia = min(s_lo[0], min(s_lo[1], s_lo[2])), ib = max(s_hi[0], max(s_hi[1], s_hi[2]));
  const int nrow = ib - ia + 1;
  if (nrow <= 0) return;
  const int Ya = lo + ia;
  const int xg = col_tile * tw + (int)threadIdx.x % tw, rphase = (int)threadIdx.x / tw;
  if (xg >= wv || rphase >= rp) return;
  const int X = xg * VEC;
  const int k1 = min(k + 1, h - 1);
  const float* r0 = in + (size_t)plane * h * w + (size_t)k * w;
  const float* r1 = in + (size_t)plane * h * w + (size_t)k1 * w;
  float t0[VEC], t1[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const Tap tx = bilinear_tap(min(X + i, W - 1), scale_w, w, W);
    t0[i] = __fmaf_rn(__ldg(r0 + tx.i0), tx.w0, __fmul_rn(__ldg(r0 + tx.i1), tx.w1));
    t1[i] = __fmaf_rn(__ldg(r1 + tx.i0), tx.w0, __fmul_rn(__ldg(r1 + tx.i1), tx.w1));
  }
  float* dst = out + (size_t)plane * H * W + (size_t)(Ya + rphase) * W + X;
  const size_t step = (size_t)rp * W;
#pragma unroll 4
  for (int r = rphase; r < nrow; r += rp) {
    const float h0 = s_h0[ia + r], h1 = s_h1[ia + r];
    float o[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] = __fmaf_rn(t0[i], h0, __fmul_rn(t1[i], h1));
    if (VEC == 4)
      stg_stream4(dst, make_float4(o[0], o[1], o[2], o[3]));
    else
      stg_stream1(dst, o[0]);
    dst += step;
  }
}

// Adjoint.  block = (plane, group of RY low-res rows).  Dynamic smem: colsum[RY][W] | wrow[ny_cap][RY].
//   step 0: per full-res row Y of the group's footprint, its weight towards each of the RY low-res rows
//   step 1: stream the footprint rows once (VEC=4: 128-bit loads), reduce along y in registers -> colsum
//   step 2: reduce colsum along x into the RY*w outputs
template <int RY, int VEC>
__global__ void __launch_bounds__(kUpThreads)
upsample_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gin, int h, int w, int H, int W,
                    float scale_h, float scale_w, float inv_scale_h, float inv_scale_w, int ny_cap) {
  extern __shared__ __align__(16) float up_smem[];
  float* colsum = up_smem;                 // [RY][W]
  float* wrow = up_smem + (size_t)RY * W;  // [ny_cap][RY]
  const long long plane = blockIdx.y;
  const int ybase = blockIdx.x * RY;
  const int ylast = min(ybase + RY, h) - 1;
  const float* g = gout + (size_t)plane * H * W;
  // conservative full-res row range touching low-res rows [ybase, ylast]; exact membership is decided per row
  int Ylo = (int)floorf(((float)ybase - 0.5f) * inv_scale_h - 0.5f) - 2;
  int Yhi = (int)ceilf(((float)ylast + 1.5f) * inv_scale_h - 0.5f) + 2;
  Ylo = max(Ylo, 0);
  Yhi = min(Yhi, H - 1);
  if (h == H) {
    Ylo = ybase;
    Yhi = ylast;
  }
  Yhi = min(Yhi, Ylo + ny_cap - 1);  // ny_cap is sized by the host to cover the footprint
  const int ny = Yhi - Ylo + 1;
  for (int i = threadIdx.x; i < ny; i += kUpThreads) {
    const Tap ty = bilinear_tap(Ylo + i, scale_h, h, H);
#pragma unroll
    for (int r = 0; r < RY; ++r) {
      float wgt = 0.f;
      if (ty.i0 - ybase == r) wgt += ty.w0;
      if (ty.i1 - ybase == r) wgt += ty.w1;
      wrow[i * RY + r] = wgt;
    }
  }
  for (int i = threadIdx.x; i < RY * W; i += kUpThreads) colsum[i] = 0.f;
  __syncthreads();
  const int ngroups = (W + VEC - 1) / VEC;                  // column groups per row
  const int nsplit = max(1, min(kUpThreads / ngroups, 8));  // row-interleaved thread teams per column group
  const int team = threadIdx.x / ngroups;
  const bool working = team < nsplit || ngroups >= kUpThreads;
  for (int g0 = 0; g0 < ngroups; g0 += kUpThreads) {
    const int xg = g0 + (ngroups >= kUpThreads ? threadIdx.x : threadIdx.x - team * ngroups);
    float acc[RY][VEC];
#pragma unroll
    for (int r = 0; r < RY; ++r)
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[r][k] = 0.f;
    if (working && xg < ngroups) {
      const int ystep = ngroups >= kUpThreads ? 1 : nsplit;
      const float* gp = g + (size_t)Ylo * W + (size_t)xg * VEC;
#pragma unroll 4
      for (int i = (ngroups >= kUpThreads ? 0 : team); i < ny; i += ystep) {
        float v[VEC];
        if (VEC == 4) {
          const float4 t = ldg_stream4(gp + (size_t)i * W);
          v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
        } else {
          v[0] = ldg_stream1(gp + (size_t)i * W);
        }
        float wr[RY];
        if (RY == 4) {
          const float4 t = *reinterpret_cast<const float4*>(wrow + i * RY);
          wr[0] = t.x, wr[1] = t.y, wr[2] = t.z, wr[3] = t.w;
        } else {
#pragma unroll
          for (int r = 0; r < RY; ++r) wr[r] = wrow[i * RY + r];
        }
#pragma unroll
        for (int r = 0; r < RY; ++r)
#pragma unroll
          for (int k = 0; k < VEC; ++k) acc[r][k] = fmaf(wr[r], v[k], acc[r][k]);
      }
    }
    // fixed-order combination of the teams (deterministic)
    for (int s = 0; s < (ngroups >= kUpThreads ? 1 : nsplit); ++s) {
      if (working && xg < ngroups && (ngroups >= kUpThreads || team == s)) {
#pragma unroll
        for (int r = 0; r < RY; ++r)
#pragma unroll
          for (int k = 0; k < VEC; ++k) colsum[r * W + xg * VEC + k] += acc[r][k];
      }
      __syncthreads();
    }
  }
  // reduce along x: out[y][x] = sum_X wx(X,x) colsum[y][X]
  const int n_out = RY * w;
  for (int o = threadIdx.x; o < n_out; o += kUpThreads) {
    const int r = o / w, x = o - r * w;
    if (ybase + r >= h) continue;
    int Xlo = (int)floorf(((float)x - 0.5f) * inv_scale_w - 0.5f) - 2;
    int Xhi = (int)ceilf(((float)x + 1.5f) * inv_scale_w - 0.5f) + 2;
    Xlo = max(Xlo, 0);
    Xhi = min(Xhi, W - 1);
    if (w == W) Xlo = Xhi = x;
    float acc = 0.f;
    for (int X = Xlo; X <= Xhi; ++X) {
      const Tap tx = bilinear_tap(X, scale_w, w, W);
      float wgt = 0.f;
      if (tx.i0 == x) wgt += tx.w0;
      if (tx.i1 == x) wgt += tx.w1;
      acc = fmaf(wgt, colsum[r * W + X], acc);
    }
    gin[((size_t)plane * h + ybase + r) * w + x] = acc;
  }
}

// Adjoint, sweep form (integer upscale factors that are a multiple of 8 along x, rows of <= 1024 elements: the
// training shapes).  thread = 4 consecutive X, which then share one pair of x taps; blockDim = W / 4.
// Work = the planes * h low-res rows of the whole tensor, cut into gridDim.x EQUAL contiguous ranges (a range that
// crosses a plane boundary is processed as two segments), so that every SM streams the same number of bytes whatever
// the shape (24x17 planes of 32 rows and 3x151 planes alike; fixed 16-row segments left 8 % / 50 % of the SMs idle).
// A segment walks the full-res rows of its intervals top-down exactly once through a rolling window of UN 16-byte
// cp.async copies per thread that stays full across the row emits: per row 8 FMAs fold the x weights, 4 more the y
// weights; a low-res row is emitted when the sweep leaves its interval (shared-memory gather over the threads whose
// taps hit each cell, fixed order).  Nothing is read twice: the lower-tap sums of a segment's LAST interval belong to
// the next segment's first row, which therefore receives exactly two contributions - its owner's and this carry -
// added with atomicAdd onto a zeroed output.  Two operands commute, so the result does not depend on which block
// comes first: deterministic without a second pass.  (Round 2: the first sweep kernel executed 78 instructions per
// 16 bytes - ncu: 66 % issue-active, barrier + shared-memory stalls - and re-read one interval per range; a pure read
// with this access pattern reaches 6.3 TB/s once ~1500 threads per SM are streaming, scripts/read_probe.py.)
template <int UN>
__global__ void __launch_bounds__(256, 4)
upsample_bwd_sweep_kernel(const float* __restrict__ gout, float* __restrict__ gin, int h, int w, int H, int W,
                          float scale_h, float scale_w, long long total_rows, int cap_rows, int ny_cap) {
  extern __shared__ __align__(16) uint8_t up_dyn[];
  const int wv = blockDim.x;  // == W / 4
  const int tid = threadIdx.x;
  float4* ring = reinterpret_cast<float4*>(up_dyn);                       // [UN][wv]
  // 8-byte entries first: every array starts aligned whatever ny_cap and wv are
  float2* s_p = reinterpret_cast<float2*>(ring + (size_t)UN * wv);        // [2][wv] (p0, p1) of the row being emitted
  short4* s_j = reinterpret_cast<short4*>(s_p + 2 * wv);                  // [w] thread ranges hitting low-res x
  float2* s_h = reinterpret_cast<float2*>(s_j + w);                       // [ny_cap] y weights (upper tap, lower tap)
  int* s_k = reinterpret_cast<int*>(s_h + ny_cap);                        // [ny_cap] low-res row of the upper tap
  int* s_x0 = s_k + ny_cap;                                               // [wv] upper / lower x tap of each thread
  int* s_x1 = s_x0 + wv;
  __shared__ int s_lim[2];                                                // first / last+1 tap-table row actually read
  const int X = tid * 4;
  float wx0[4], wx1[4];
  sweep_x_taps(tid, wv, w, W, scale_w, wx0, wx1, s_x0, s_x1, s_j);
  const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring + tid);  // this thread's 16 B of slot 0
  const uint32_t slot_b = (uint32_t)wv * 16u;
  int flip = 0;
  // this block's range of global low-res rows (plane * h + y)
  const long long r_begin = total_rows * (long long)blockIdx.x / (long long)gridDim.x;
  const long long r_end = total_rows * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
  for (long long r = r_begin; r < r_end;) {
    const long long plane = r / h;
    const int y0 = (int)(r - plane * h);
    const int ylast = (int)min((long long)min(h, y0 + cap_rows), y0 + (r_end - r)) - 1;
    r += ylast - y0 + 1;
    int i_lo, i_hi;
    const int Ylo = sweep_y_taps(tid, wv, y0, ylast, h, H, scale_h, ny_cap, s_k, s_h, s_lim, i_lo, i_hi);
    const float* gp = gout + (size_t)plane * H * W + (size_t)(Ylo + i_lo) * W + X;  // next row to fetch
    float* out = gin + (size_t)plane * h * w;
    float a0p0 = 0.f, a0p1 = 0.f, a1p0 = 0.f, a1p1 = 0.f, c0 = 0.f, c1 = 0.f;  // current interval, carry from the one above
    int cur = -1;
    // low-res row `row` += gather over x of the per-thread pairs (v0 -> upper x tap, v1 -> lower x tap); `shared`:
    // another segment contributes to this row as well (see the header comment)
    auto emit = [&](int row, float v0, float v1, bool shared) {
      s_p[flip * wv + tid] = make_float2(v0, v1);
      __syncthreads();  // one barrier per emit: the buffers alternate, so the next emit cannot overtake this gather
      if (tid < w) {
        const short4 jr = s_j[tid];
        const float2* sp = s_p + flip * wv;
        float acc = 0.f;
        for (int j = jr.x; j < jr.y; ++j) acc += sp[j].x;
        for (int j = jr.z; j < jr.w; ++j) acc += sp[j].y;
        if (shared)
          atomicAdd(out + (size_t)row * w + tid, acc);
        else
          out[(size_t)row * w + tid] = acc;
      }
      flip ^= 1;
    };
    // leave interval `cur`: emit low-res row cur, its lower-tap sums become the carry
    auto flush = [&]() {
      emit(cur, a0p0 + c0, a0p1 + c1, cur == y0 && y0 > 0);
      c0 = a1p0, c1 = a1p1;
      a0p0 = a0p1 = a1p0 = a1p1 = 0.f;
    };
    // rolling window of UN rows in flight per thread: cp.async into the thread's own 16 B of ring slot (row % UN) (a
    // thread only ever reads what it copied itself: no block barrier, just its own wait_group)
    int nfetch = i_hi - i_lo;  // rows still to fetch
    uint32_t fslot = 0, cslot = 0;
    auto fetch = [&]() {
      if (nfetch > 0) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ring_s + fslot), "l"(gp) : "memory");
        gp += W;
        --nfetch;
      }
      cp_async_commit();
      fslot = (fslot + slot_b == slot_b * UN) ? 0u : fslot + slot_b;
    };
#pragma unroll
    for (int j = 0; j < UN - 1; ++j) fetch();
#pragma unroll 1
    for (int i = i_lo; i < i_hi; ++i) {
      fetch();
      cp_async_wait<UN - 1>();
      const int k = s_k[i];
      if (k != cur) {  // uniform over the block
        if (cur >= 0) flush();
        cur = k;
      }
      float4 x;
      asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "r"(ring_s + cslot));
      cslot = (cslot + slot_b == slot_b * UN) ? 0u : cslot + slot_b;
      const float2 hw = s_h[i];
      const float p0 = fmaf(x.w, wx0[3], fmaf(x.z, wx0[2], fmaf(x.y, wx0[1], x.x * wx0[0])));
      const float p1 = fmaf(x.w, wx1[3], fmaf(x.z, wx1[2], fmaf(x.y, wx1[1], x.x * wx1[0])));
      a0p0 = fmaf(hw.x, p0, a0p0), a0p1 = fmaf(hw.x, p1, a0p1);
      a1p0 = fmaf(hw.y, p0, a1p0), a1p1 = fmaf(hw.y, p1, a1p1);
    }
    cp_async_wait<0>();
    if (cur >= 0) {
      flush();
      if (ylast < h - 1) emit(ylast + 1, c0, c1, true);  // lower-tap sums of the last interval: the next segment's row
    }
  }
}

// Prediction without the upsample: pred[b,Y,X] = argmax over c of the value ucd_upsample_bilinear_fwd writes at
// [b,c,Y,X], bit for bit: the same taps and the same bilinear_blend operation order (SMALL: ATen's small-output order,
// H + W <= 128), ties to the first maximal channel, NaN maximal (torch.argmax).  block = (image, low-res row interval
// k, column tile); thread (x, g) owns column x and rows g, g + kArgRG, ... of the interval, kArgRPT of them per pass
// (intervals longer than kArgRG * kArgRPT rows, i.e. scale factors above ~30, take more passes).  Channels are the
// outer loop: the column's 2x2 source cell is loaded once per channel and every row of the thread updates a running
// (max, index) held in registers.  Only the int64 prediction is written.
constexpr int kArgTX = 64, kArgRG = 4, kArgRPT = 8;
template <bool SMALL>
__global__ void __launch_bounds__(kArgTX * kArgRG)
upsample_argmax_kernel(const float* __restrict__ in, int64_t* __restrict__ pred, int C, int h, int w, int H, int W,
                       float scale_h, float scale_w) {
  __shared__ int s_ya, s_yb;
  const int b = blockIdx.z, k = blockIdx.y;
  const int xl = threadIdx.x % kArgTX, rg = threadIdx.x / kArgTX;  // rg is warp-uniform
  const int X = blockIdx.x * kArgTX + xl;
  // rows of this interval: all Y with tap.i0 == k (contiguous), found in a conservative candidate range
  if (threadIdx.x == 0) s_ya = H, s_yb = -1;
  __syncthreads();
  const float inv = (float)H / (float)h;
  const int lo = max((int)floorf(((float)k - 0.5f) * inv) - 2, 0);
  const int hi = min((int)ceilf(((float)k + 1.5f) * inv) + 2, H - 1);
  for (int Y = lo + (int)threadIdx.x; Y <= hi; Y += blockDim.x)
    if (bilinear_tap(Y, scale_h, h, H).i0 == k) atomicMin(&s_ya, Y), atomicMax(&s_yb, Y);
  __syncthreads();
  const int Ya = s_ya, nrow = s_yb - s_ya + 1;
  if (nrow <= 0 || X >= W) return;
  const Tap tx = bilinear_tap(X, scale_w, w, W);
  const int k1 = min(k + 1, h - 1);  // = the lower tap of every row of the interval
  const int o00 = k * w + tx.i0, o01 = k * w + tx.i1, o10 = k1 * w + tx.i0, o11 = k1 * w + tx.i1;
  const size_t plane = (size_t)h * w;
  const float* src = in + (size_t)b * C * plane;
  for (int r0 = rg; r0 < nrow; r0 += kArgRG * kArgRPT) {
    const int nj = (nrow - r0 + kArgRG - 1) / kArgRG;  // rows of this thread in this pass (warp-uniform)
    float h0[kArgRPT], h1[kArgRPT], best[kArgRPT];
    int arg[kArgRPT];
#pragma unroll
    for (int j = 0; j < kArgRPT; ++j) {
      const Tap ty = bilinear_tap(Ya + min(r0 + j * kArgRG, nrow - 1), scale_h, h, H);
      h0[j] = ty.w0, h1[j] = ty.w1, best[j] = -INFINITY, arg[j] = 0;
    }
    const float* p = src;
    for (int c = 0; c < C; ++c, p += plane) {
      const float v00 = __ldg(p + o00), v01 = __ldg(p + o01), v10 = __ldg(p + o10), v11 = __ldg(p + o11);
#pragma unroll
      for (int j = 0; j < kArgRPT; ++j) {
        if (!SMALL && j >= nj) break;  // (with this exit the SMALL form, 4 weight products per row, spills registers)
        const float v = bilinear_blend(SMALL, v00, v01, v10, v11, h0[j], h1[j], tx.w0, tx.w1);
        if (j < nj && (v > best[j] || (isnan(v) && !isnan(best[j])))) best[j] = v, arg[j] = c;
      }
    }
#pragma unroll
    for (int j = 0; j < kArgRPT; ++j)
      if (j < nj) pred[((size_t)b * H + Ya + r0 + j * kArgRG) * W + X] = arg[j];
  }
}

}  // namespace ucd

using namespace ucd;

extern "C" int ucd_upsample_bilinear_fwd(const float* in, float* out, int64_t planes, int h, int w, int H, int W,
                                         void* stream) {
  UCD_CHECK_ARG(in && out, "ucd_upsample_bilinear_fwd: null pointer");
  UCD_CHECK_ARG(planes > 0 && h > 0 && w > 0 && H > 0 && W > 0, "ucd_upsample_bilinear_fwd: bad shape");
  UCD_CHECK_ARG((long long)h * w < (1ll << 30), "ucd_upsample_bilinear_fwd: source plane too large");
  cudaStream_t st = (cudaStream_t)stream;
  const float sh = (float)h / (float)H, sw = (float)w / (float)W;
  const bool v4 = (W % 4 == 0) && aligned16(out);
  const int wv = v4 ? W / 4 : W;
  // upsampling beyond ATen's small-output regime (every training shape): interval kernel
  if (H + W > 128 && H >= h && W >= w && (double)H / h <= 40.0 /* candidate rows per interval: 2*scale + 5 <= kUpMaxIvRows */ && planes * (long long)h < (1ll << 30) / 64) {
    const int tw = wv < kUpThreads ? wv : kUpThreads;
    const int nct = (wv + tw - 1) / tw;
    const unsigned nblk = (unsigned)(planes * h * nct);
    if (v4)
      upsample_fwd_interval_kernel<4><<<nblk, kUpThreads, 0, st>>>(in, out, h, w, H, W, sh, sw, tw, nct);
    else
      upsample_fwd_interval_kernel<1><<<nblk, kUpThreads, 0, st>>>(in, out, h, w, H, W, sh, sw, tw, nct);
    UCD_CHECK_LAUNCH("upsample_fwd_interval_kernel");
    return UCD_OK;
  }
  const long long work = (long long)H * wv;
  const int gx = (int)((work + kUpThreads - 1) / kUpThreads);
  // planes per block: enough to amortise the tap computation (>= 16 planes when there are that many), few enough
  // that the grid is many waves deep (blocks finish at different times; a 2-3 wave grid left SMs idle)
  long long want_y = (32ll * kNumSMs + gx - 1) / gx;
  if (want_y < 1) want_y = 1;
  if (want_y > (planes + 15) / 16) want_y = (planes + 15) / 16;
#ifdef UCD_DEBUG_KNOBS
  if (const char* e = getenv("UCD_UP_GY")) want_y = atoi(e) > 0 ? atoi(e) : want_y;  // tuning knob
#endif
  if (want_y > planes) want_y = planes;
  const int ppb = (int)((planes + want_y - 1) / want_y);
  const int gy = (int)((planes + ppb - 1) / ppb);
  UCD_CHECK_ARG(gy <= 65535, "ucd_upsample_bilinear_fwd: too many planes");
  dim3 grid(gx, gy);
  if (v4)
    upsample_fwd_kernel<4><<<grid, kUpThreads, 0, st>>>(in, out, planes, h, w, H, W, sh, sw, ppb);
  else
    upsample_fwd_kernel<1><<<grid, kUpThreads, 0, st>>>(in, out, planes, h, w, H, W, sh, sw, ppb);
  UCD_CHECK_LAUNCH("upsample_fwd_kernel");
  return UCD_OK;
}

extern "C" int ucd_upsample_bilinear_bwd(const float* gout, float* gin, int64_t planes, int h, int w, int H, int W,
                                         void* stream) {
  UCD_CHECK_ARG(gout && gin, "ucd_upsample_bilinear_bwd: null pointer");
  UCD_CHECK_ARG(planes > 0 && h > 0 && w > 0 && H > 0 && W > 0, "ucd_upsample_bilinear_bwd: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  constexpr int RY = 4;
  // full-res rows that can touch RY consecutive low-res rows (+ the slack the kernel adds around its estimate)
  const int ny_cap = (h == H) ? RY : (int)((double)(RY + 2) * H / h) + 8;
  const size_t smem = ((size_t)RY * W + (size_t)ny_cap * RY) * sizeof(float);
  UCD_CHECK_ARG(smem <= 200 * 1024, "ucd_upsample_bilinear_bwd: W=%d / scale too large for one block", W);
  const float sh = (float)h / (float)H, sw = (float)w / (float)W;
  const bool v4 = (W % 4 == 0) && aligned16(gout);
  // sweep form: integer scales, a multiple of 8 along x (4 consecutive X share their taps), one block row = W/4 threads.
  // Grid = a whole number of blocks per SM (~1500 streaming threads per SM), each with an equal share of the
  // planes * h low-res rows; small problems take fewer blocks so that a range keeps >= 4 rows.
  const int up = H / (h > 0 ? h : 1);
  constexpr int kUpSweepTaps = 640;  // tap-table rows a block may hold
  const int cap_rows = up > 0 ? (kUpSweepTaps - 8) / up - 2 : 0;  // rows of one segment the tap table can hold
  if (v4 && H % h == 0 && W % w == 0 && (W / w) % 8 == 0 && W / 4 <= 256 && (W / 4) % 32 == 0 && w <= W / 4 &&
      cap_rows >= 1) {
    int un = 8, bps = (W / 4 <= 128 ? 4 : 2);  // rows in flight per thread, blocks per SM (measured best: scripts/up_bwd_probe.py)
#ifdef UCD_DEBUG_KNOBS
    if (const char* e = getenv("UCD_UPB_UN")) un = atoi(e);    // tuning knobs (debug library only)
    if (const char* e = getenv("UCD_UPB_BPS")) bps = atoi(e);
#endif
    const long long total_rows = planes * h;
    long long nb = (long long)kNumSMs * bps;
    while (nb > kNumSMs && total_rows / nb < 4) nb -= kNumSMs;
    if (nb > total_rows) nb = total_rows;
    long long seg = (total_rows + nb - 1) / nb + 1;  // longest segment of a range
    if (seg > cap_rows) seg = cap_rows;
    const int ny_cap = (int)(seg + 2) * up + 8;
    const int wv4 = W / 4;
    const size_t dyn = (size_t)un * wv4 * 16 + (size_t)2 * wv4 * 8 + (size_t)ny_cap * 12 + (size_t)2 * wv4 * 4 + (size_t)w * 8;
    // boundary rows of the ranges are accumulated by two blocks (see the kernel): the output starts from zero
    cudaError_t e = cudaMemsetAsync(gin, 0, (size_t)planes * h * w * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(upsample_bwd)");
    auto kern = upsample_bwd_sweep_kernel<8>;
#ifdef UCD_DEBUG_KNOBS
    if (un == 4) kern = upsample_bwd_sweep_kernel<4>;
    if (un == 12) kern = upsample_bwd_sweep_kernel<12>;
    if (un == 16) kern = upsample_bwd_sweep_kernel<16>;
#endif
    if (dyn > 48 * 1024) {
      e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(upsample_bwd_sweep)");
    }
    kern<<<(unsigned)nb, wv4, dyn, st>>>(gout, gin, h, w, H, W, sh, sw, total_rows, cap_rows, ny_cap);
    UCD_CHECK_LAUNCH("upsample_bwd_sweep_kernel");
    return UCD_OK;
  }
  auto kern = v4 ? upsample_bwd_kernel<RY, 4> : upsample_bwd_kernel<RY, 1>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(upsample_bwd)");
  }
  const int gyb = (h + RY - 1) / RY;
  for (int64_t p0 = 0; p0 < planes; p0 += 65535) {  // grid.y limit
    const int np = (int)((planes - p0 < 65535) ? planes - p0 : 65535);
    dim3 grid(gyb, np);
    kern<<<grid, kUpThreads, smem, st>>>(gout + (size_t)p0 * H * W, gin + (size_t)p0 * h * w, h, w, H, W, sh, sw,
                                         (float)H / (float)h, (float)W / (float)w, ny_cap);
    UCD_CHECK_LAUNCH("upsample_bwd_kernel");
  }
  return UCD_OK;
}

extern "C" int ucd_upsample_argmax(const float* lr, int64_t* pred, int B, int C, int h, int w, int H, int W,
                                   void* stream) {
  UCD_CHECK_ARG(lr && pred, "ucd_upsample_argmax: null pointer");
  UCD_CHECK_ARG(B > 0 && C > 0 && h > 0 && w > 0 && H >= h && W >= w, "ucd_upsample_argmax: bad shape (upsampling only)");
  UCD_CHECK_ARG(B <= 65535 && h <= 65535, "ucd_upsample_argmax: batch / rows too large for the grid");
  UCD_CHECK_ARG((long long)h * w < (1ll << 30), "ucd_upsample_argmax: source plane too large");
  cudaStream_t st = (cudaStream_t)stream;
  const float sh = (float)h / (float)H, sw = (float)w / (float)W;
  dim3 grid((W + kArgTX - 1) / kArgTX, h, B);
  if (H + W <= 128)  // the operation order ucd_upsample_bilinear_fwd uses at this size
    upsample_argmax_kernel<true><<<grid, kArgTX * kArgRG, 0, st>>>(lr, pred, C, h, w, H, W, sh, sw);
  else
    upsample_argmax_kernel<false><<<grid, kArgTX * kArgRG, 0, st>>>(lr, pred, C, h, w, H, W, sh, sw);
  UCD_CHECK_LAUNCH("upsample_argmax_kernel");
  return UCD_OK;
}
