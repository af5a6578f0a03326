// MiB unbiased cross-entropy and unbiased knowledge distillation, forward and backward.
// Reference semantics: utils/loss.py:96-109 (UnbiasedCrossEntropy.forward) and
// utils/loss.py:148-184 (UnbiasedKnowledgeDistillationLoss.forward); closed forms and gradients
// in SURVEY.md Appendix A.3.
//
// All four kernels are HBM-bound streaming kernels over NCHW fp32 logits: a thread owns VEC
// consecutive pixels (VEC=4 -> 128-bit coalesced accesses, a warp touches 512 contiguous bytes per
// channel), walks the C channels with stride H*W and keeps every log-sum-exp it needs as an online
// (max, sum) pair in registers, so x (and t) are read exactly once per pass.  One MUFU.EX2 per
// element (see lse_push).  Partial sums go to a per-block slot and are reduced by a second
// fixed-order kernel, so results are run-to-run deterministic.
#include "common.cuh"
#include "sweep_adjoint.cuh"

#include <stdlib.h>

namespace ucd {

constexpr int kStreamThreads = 256;
constexpr int kStreamMaxBlocks = kNumSMs * 8;
constexpr int kScratchFloats = 4 * kStreamMaxBlocks + 64;

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    float4 t = ldg_stream4(p);
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  }
  static __device__ __forceinline__ void load_cached(const float* p, float (&v)[4]) {
    float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
  static __device__ __forceinline__ void store_stream(float* p, const float (&v)[4]) {
    stg_stream4(p, make_float4(v[0], v[1], v[2], v[3]));
  }
};
template <>
struct Vec<1> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[1]) { v[0] = ldg_stream1(p); }
  static __device__ __forceinline__ void load_cached(const float* p, float (&v)[1]) { v[0] = *p; }
  static __device__ __forceinline__ void store(float* p, const float (&v)[1]) { *p = v[0]; }
  static __device__ __forceinline__ void store_stream(float* p, const float (&v)[1]) { stg_stream1(p, v[0]); }
};

// dx store of the backward kernels.  ACC: add to what is already there - the second of two losses on the same logits
// accumulates into the first one's gradient buffer, so autograd never runs its own add kernel over two full-size
// gradients (ucd_b200/losses.py::_GradSlot; it was 8 % of the drop-in step).
template <int VEC, bool ACC>
__device__ __forceinline__ void store_dx(float* p, float (&o)[VEC]) {
  if (ACC) {
    float old[VEC];
    Vec<VEC>::load(p, old);
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] += old[i];
  }
  Vec<VEC>::store_stream(p, o);
}

// fixed-order final reduction of per-block partial sums: out[k] = sum_b part[k*nblk + b]
__global__ void reduce_partials_kernel(const float* __restrict__ part, int nblk, int nk, float* __restrict__ out,
                                       float scale) {
  __shared__ float red[32];
  for (int k = 0; k < nk; ++k) {
    float acc = 0.f;
    for (int i = threadIdx.x; i < nblk; i += blockDim.x) acc += part[(size_t)k * nblk + i];
    float r = block_sum(acc, red);
    if (threadIdx.x == 0) out[k] = r * scale;
  }
}

constexpr float kNegBig = -3.0e38f;
constexpr int kLseChunk = 8;

// Online log-sum-exp (log2 domain) of channels [c0,c1) of VEC adjacent pixels, kLseChunk channels at a time.
// PICK: also fetch x[label] on the way.
template <int VEC, bool PICK>
__device__ __forceinline__ void lse_chunks(const float* __restrict__ xp, long long HW, int c0, int c1,
                                           const long long (&lab)[VEC], float (&m)[VEC], float (&s)[VEC],
                                           float (&picked)[VEC]) {
  for (int c = c0; c < c1; c += kLseChunk) {
    float v[kLseChunk][VEC];
#pragma unroll
    for (int k = 0; k < kLseChunk; ++k) {
      if (c + k < c1) {
        Vec<VEC>::load(xp + (long long)(c + k) * HW, v[k]);
      } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) v[k][i] = kNegBig;
      }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float cm = v[0][i];
#pragma unroll
      for (int k = 1; k < kLseChunk; ++k) cm = fmaxf(cm, v[k][i]);
      const float nm = fmaxf(m[i], cm * kLog2e);
      float acc = s[i] * ex2f(m[i] - nm);
#pragma unroll
      for (int k = 0; k < kLseChunk; ++k) {
        acc += ex2f(fmaf(v[k][i], kLog2e, -nm));
        if (PICK) picked[i] = (lab[i] == c + k) ? v[k][i] : picked[i];
      }
      m[i] = nm;
      s[i] = acc;
    }
  }
}

// ------------------------------------------------------------------------------------------
// UNCE forward
// ------------------------------------------------------------------------------------------
// A thread owns VEC adjacent pixels and walks the channels in chunks of 4 with ONE pointer that advances by 4 planes:
// 4 independent 128-bit loads, then per pixel the chunk maximum rescales the running sum once (5 exps per 4 elements).
// Old classes first, then the rest; the running log-sum-exp is snapshotted where the groups meet (lse over the old
// classes).  x[label] is fetched by its own 4-byte load up front instead of a compare + select per element.
// Round 2: the first version of this loop executed 37 thread instructions per logit (64-bit index arithmetic, range
// predicates and label compares per element; ncu: 62 % issue-active at 5.1 TB/s) - it was issue-bound, not memory-
// bound.  This form needs ~6 per element and 64 registers (4 blocks per SM: a pure read of the same planes reaches
// 6.3 TB/s with 1024 threads per SM and 4 loads in flight per thread, scripts/read_probe.py).
template <int VEC>
__device__ __forceinline__ void lse_chunk4(const float (&v)[4][VEC], float (&m)[VEC], float (&s)[VEC]) {
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const float cm = fmaxf(fmaxf(v[0][i], v[1][i]), fmaxf(v[2][i], v[3][i]));
    const float nm = fmaxf(m[i], cm * kLog2e);
    float acc = s[i] * ex2f(m[i] - nm);
#pragma unroll
    for (int k = 0; k < 4; ++k) acc += ex2f(fmaf(v[k][i], kLog2e, -nm));
    m[i] = nm;
    s[i] = acc;
  }
}

// online log-sum-exp (log2 domain) of the next n planes at xc (plane stride HW); xc advances past them
template <int VEC>
__device__ __forceinline__ void lse_planes(const float*& xc, long long HW, int n, float (&m)[VEC], float (&s)[VEC]) {
  int c = 0;
  for (; c + 4 <= n; c += 4) {
    float v[4][VEC];
    Vec<VEC>::load(xc, v[0]);
    Vec<VEC>::load(xc + HW, v[1]);
    Vec<VEC>::load(xc + 2 * HW, v[2]);
    Vec<VEC>::load(xc + 3 * HW, v[3]);
    xc += 4 * HW;
    lse_chunk4<VEC>(v, m, s);
  }
  if (c < n) {  // 1-3 planes left: the missing ones count as -inf
    float v[4][VEC];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (c + k < n) {
        Vec<VEC>::load(xc + k * HW, v[k]);
      } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) v[k][i] = kNegBig;
      }
    }
    xc += (long long)(n - c) * HW;
    lse_chunk4<VEC>(v, m, s);
  }
}

// (image, first pixel) of pixel group g; 32-bit arithmetic whenever the group count allows it
__device__ __forceinline__ void group_to_bp(long long g, long long gpi, bool small, int vec, long long& b, long long& p) {
  if (small) {
    const unsigned bb = (unsigned)g / (unsigned)gpi;
    b = bb;
    p = (long long)((unsigned)g - bb * (unsigned)gpi) * vec;
  } else {
    b = g / gpi;
    p = (g - b * gpi) * vec;
  }
}

template <int VEC>
__global__ void __launch_bounds__(kStreamThreads, VEC == 4 ? 4 : 2)
unce_fwd_kernel(const float* __restrict__ x, long long* __restrict__ y, float* __restrict__ loss_px,
                float* __restrict__ lse_all_out, float* __restrict__ lse_old_out, float* __restrict__ part,
                int B, int C, int old_cl, long long HW, int ignore_index) {
  const long long gpi = HW / VEC;  // groups per image
  const long long n_groups = gpi * B;
  const bool small = n_groups < (1ll << 31) && gpi < (1ll << 31);
  const int oc = old_cl < C ? (old_cl > 0 ? old_cl : 0) : C;
  float loss_acc = 0.f, valid_acc = 0.f;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups;
       g += (long long)gridDim.x * blockDim.x) {
    long long b, p;
    group_to_bp(g, gpi, small, VEC, b, p);
    const float* xp = x + (b * C) * HW + p;
    long long* yp = y + b * HW + p;
    long long yl[VEC];
    if (VEC == 4) {
      const longlong2 t0 = *reinterpret_cast<const longlong2*>(yp), t1 = *reinterpret_cast<const longlong2*>(yp + 2);
      yl[0] = t0.x, yl[1] = t0.y, yl[2 % VEC] = t1.x, yl[3 % VEC] = t1.y;
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) yl[i] = yp[i];
    }
    int lab[VEC];
    float picked[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      long long t = yl[i];
      if (t < old_cl) {  // loss.py:104-105: labels[targets < old_cl] = 0 (in place)
        if (t != 0) yp[i] = 0;
        t = 0;
      }
      lab[i] = (t < 0 || t > 0x7fffffffLL) ? -1 : (int)t;  // out-of-range labels can never match a channel
      // x[label]: its own load, issued before the planes are streamed (the sector is read again by the stream: L2 hit)
      picked[i] = (lab[i] >= 0 && lab[i] < C) ? __ldg(xp + (long long)lab[i] * HW + i) : 0.f;
    }
    float m[VEC], s[VEC], lse_old2[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) m[i] = kNegBig, s[i] = 0.f;
    const float* xc = xp;
    lse_planes<VEC>(xc, HW, oc, m, s);
#pragma unroll
    for (int i = 0; i < VEC; ++i) lse_old2[i] = m[i] + lg2f(s[i]);  // what has been summed so far: the old classes
    lse_planes<VEC>(xc, HW, C - oc, m, s);
    float out[VEC], la[VEC], lo[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float lse2 = m[i] + lg2f(s[i]);
      la[i] = lse2 * kLn2;
      lo[i] = lse_old2[i] * kLn2;
      const bool ign = lab[i] == ignore_index;
      float l = (lab[i] == 0 && old_cl > 0) ? (la[i] - lo[i]) : (la[i] - picked[i]);
      // labels outside [0,C) that are not ignore_index are a caller error (nll_loss asserts); give 0
      if (ign || lab[i] < 0 || lab[i] >= C) l = 0.f;
      out[i] = l;
      loss_acc += l;
      valid_acc += ign ? 0.f : 1.f;
    }
    Vec<VEC>::store(loss_px + b * HW + p, out);
    Vec<VEC>::store(lse_all_out + b * HW + p, la);
    if (lse_old_out != nullptr) Vec<VEC>::store(lse_old_out + b * HW + p, lo);
  }
  if (part != nullptr) {
    __shared__ float red[32];
    float r0 = block_sum(loss_acc, red);
    float r1 = block_sum(valid_acc, red);
    if (threadIdx.x == 0) {
      part[blockIdx.x] = r0;
      part[gridDim.x + blockIdx.x] = r1;
    }
  }
}

// UNCE backward:  dx_c = g * [y != ignore] * ( softmax(x)_c - (y==0 ? [c<old] exp(x_c - lse_old) : [c==y]) )
template <int VEC, bool ACC>
__global__ void __launch_bounds__(kStreamThreads)
unce_bwd_kernel(const float* __restrict__ x, const long long* __restrict__ y, const float* __restrict__ lse_all,
                const float* __restrict__ bkg_gap, const float* __restrict__ g_px,
                const float* __restrict__ g_scalar, float g_mul, const float* __restrict__ stats,
                int mean_over_valid, float* __restrict__ dx, int B, int C, int old_cl, long long HW,
                int ignore_index) {
  const long long gpi = HW / VEC;
  const long long n_groups = gpi * B;
  float gs = 0.f;
  if (g_px == nullptr) {
    gs = g_scalar[0] * g_mul;
    if (mean_over_valid) gs = gs / stats[1];
  }
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups;
       g += (long long)gridDim.x * blockDim.x) {
    const long long b = g / gpi, p = (g - b * gpi) * VEC;
    const float* xp = x + (b * C) * HW + p;
    float* dp = dx + (b * C) * HW + p;
    const long long* yp = y + b * HW + p;
    float la2[VEC], up[VEC], fold[VEC];
    int lab[VEC];
    {
      float la[VEC], lo[VEC], gp[VEC];
      Vec<VEC>::load_cached(lse_all + b * HW + p, la);
      Vec<VEC>::load_cached(bkg_gap + b * HW + p, lo);  // lse_all - lse_old where the label is 0 (the forward's loss_px)
      if (g_px != nullptr) Vec<VEC>::load_cached(g_px + b * HW + p, gp);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        long long t = yp[i];
        if (t < old_cl) t = 0;
        const bool dead = (t == ignore_index) || t < 0 || t >= C;
        lab[i] = dead ? -1 : (int)t;
        up[i] = dead ? 0.f : (g_px != nullptr ? gp[i] : gs);
        la2[i] = la[i] * kLog2e;
        // exp(x - lse_old) = exp(x - lse_all) * exp(lse_all - lse_old); only read where the label is 0
        fold[i] = ex2f(lo[i] * kLog2e);
      }
    }
#pragma unroll 4
    for (int c = 0; c < C; ++c) {
      float v[VEC], o[VEC];
      Vec<VEC>::load(xp + (long long)c * HW, v);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float pr = ex2f(fmaf(v[i], kLog2e, -la2[i]));
        float sub;
        if (lab[i] == 0 && old_cl > 0)
          sub = (c < old_cl) ? pr * fold[i] : 0.f;
        else
          sub = (c == lab[i]) ? 1.f : 0.f;
        o[i] = up[i] * (pr - sub);
      }
      store_dx<VEC, ACC>(dp + (long long)c * HW, o);
    }
  }
}

// ------------------------------------------------------------------------------------------
// UNKD forward:  q = softmax(alpha t);  S_b = {0} U {C_old..C-1}
//   loss_px = [ q0 (lse_b - lse) + sum_{1<=c<C_old} q_c (x_c - lse) ] / C_old
// ------------------------------------------------------------------------------------------
// One chunk of 4 old-class planes of x (v) and t (u) into the running statistics of VEC pixels:
//   x: log-sum-exp (m, s);  t: log-sum-exp of alpha*t (mt, st) and wx = sum_{c>=1} 2^(alpha t_c - mt) x_c.
// nv < 4 (TAIL): only planes [0, nv) exist; skip0: plane 0 of this chunk is channel 0 (not part of wx).
template <int VEC, bool TAIL>
__device__ __forceinline__ void unkd_old_chunk(const float (&v)[4][VEC], const float (&u)[4][VEC], int nv, bool skip0,
                                               float a2, float (&m)[VEC], float (&s)[VEC], float (&mt)[VEC],
                                               float (&st)[VEC], float (&wx)[VEC]) {
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    float cm = v[0][i], ct = u[0][i] * a2;
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      const bool live = !TAIL || k < nv;
      cm = live ? fmaxf(cm, v[k][i]) : cm;
      ct = live ? fmaxf(ct, u[k][i] * a2) : ct;
    }
    const float nm = fmaxf(m[i], cm * kLog2e), nt = fmaxf(mt[i], ct);
    float acc = s[i] * ex2f(m[i] - nm);
    const float rs = ex2f(mt[i] - nt);
    float tacc = st[i] * rs, wacc = wx[i] * rs;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const bool live = !TAIL || k < nv;
      const float ex = ex2f(fmaf(v[k][i], kLog2e, -nm));
      const float et = ex2f(fmaf(u[k][i], a2, -nt));
      acc += live ? ex : 0.f;
      tacc += live ? et : 0.f;
      const float w = (live && !(k == 0 && skip0)) ? et : 0.f;
      wacc = fmaf(w, v[k][i], wacc);
    }
    m[i] = nm, s[i] = acc, mt[i] = nt, st[i] = tacc, wx[i] = wacc;
  }
}

// Round 2 rewrite (same reasons as unce_fwd_kernel above: the first version ran 66 % issue-active with 128 registers
// and two blocks per SM): one advancing pointer per tensor, chunks of 4 planes, the channels beyond the old classes
// go into their OWN (max, sum) pair - one exp per element instead of two - and lse over all channels / over the
// background set {0} U {C_old..} are combined from the pairs at the end.
template <int VEC>
__global__ void __launch_bounds__(kStreamThreads, VEC == 4 ? 3 : 2)
unkd_fwd_kernel(const float* __restrict__ x, const float* __restrict__ t, const float* __restrict__ mask,
                float alpha, float* __restrict__ out_px, float* __restrict__ lse3, float* __restrict__ part,
                int B, int C, int Cs, int C_old, int mask_zero, long long HW) {
  // C: channels of x that take part; Cs >= C: channels per image in memory (plain KD narrows x to C = C_old)
  // mask_zero: the weight of a pixel is [mask == 0] (MaskKnowledgeDistillationLoss) instead of mask itself
  const long long gpi = HW / VEC;
  const long long n_groups = gpi * B;
  const bool small = n_groups < (1ll << 31) && gpi < (1ll << 31);
  const long long plane = (long long)B * HW;
  const float a2 = alpha * kLog2e;
  const float inv_cold = 1.f / (float)C_old;
  float acc = 0.f;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups;
       g += (long long)gridDim.x * blockDim.x) {
    long long b, p;
    group_to_bp(g, gpi, small, VEC, b, p);
    const float* xp = x + (b * Cs) * HW + p;
    const float* xc = xp;
    const float* tc = t + (b * C_old) * HW + p;
    float m[VEC], s[VEC], mt[VEC], st[VEC], wx[VEC], x0[VEC], t0[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) m[i] = mt[i] = kNegBig, s[i] = st[i] = wx[i] = 0.f;
    int c = 0;
    for (; c + 4 <= C_old; c += 4) {
      float v[4][VEC], u[4][VEC];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        Vec<VEC>::load(xc + k * HW, v[k]);
        Vec<VEC>::load(tc + k * HW, u[k]);
      }
      xc += 4 * HW, tc += 4 * HW;
      if (c == 0) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) x0[i] = v[0][i], t0[i] = u[0][i] * a2;
      }
      unkd_old_chunk<VEC, false>(v, u, 4, c == 0, a2, m, s, mt, st, wx);
    }
    if (c < C_old) {  // 1-3 old planes left
      const int nv = C_old - c;
      float v[4][VEC], u[4][VEC];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k < nv) {
          Vec<VEC>::load(xc + k * HW, v[k]);
          Vec<VEC>::load(tc + k * HW, u[k]);
        } else {
#pragma unroll
          for (int i = 0; i < VEC; ++i) v[k][i] = 0.f, u[k][i] = 0.f;
        }
      }
      if (c == 0) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) x0[i] = v[0][i], t0[i] = u[0][i] * a2;
      }
      unkd_old_chunk<VEC, true>(v, u, nv, c == 0, a2, m, s, mt, st, wx);
    }
    // channels beyond the old classes: their own (max, sum) pair
    float mn[VEC], sn[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) mn[i] = kNegBig, sn[i] = 0.f;
    xc = xp + (long long)C_old * HW;
    lse_planes<VEC>(xc, HW, C - C_old, mn, sn);
    float o[VEC], l_all[VEC], l_bkg[VEC], l_t[VEC];
    float mk[VEC];
    if (mask != nullptr) Vec<VEC>::load_cached(mask + b * HW + p, mk);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      // all channels = old pair + new pair; background set = {channel 0} + new pair
      const float ma = fmaxf(m[i], mn[i]);
      const float lse2 = ma + lg2f(fmaf(s[i], ex2f(m[i] - ma), sn[i] * ex2f(mn[i] - ma)));
      const float x02 = x0[i] * kLog2e;
      const float mb = fmaxf(x02, mn[i]);
      const float lseb2 = mb + lg2f(fmaf(sn[i], ex2f(mn[i] - mb), ex2f(x02 - mb)));
      const float lset2 = mt[i] + lg2f(st[i]);
      l_all[i] = lse2 * kLn2;
      l_bkg[i] = lseb2 * kLn2;
      l_t[i] = lset2 * kLn2;
      const float q0 = ex2f(t0[i] - lset2);
      const float dot = wx[i] / st[i];  // sum_{c>=1} q_c x_c
      float l = (q0 * (l_bkg[i] - l_all[i]) + dot - (1.f - q0) * l_all[i]) * inv_cold;
      if (mask != nullptr) l *= mask_zero ? (mk[i] == 0.f ? 1.f : 0.f) : mk[i];
      o[i] = -l;
      acc += l;
    }
    if (out_px != nullptr) Vec<VEC>::store(out_px + b * HW + p, o);
    Vec<VEC>::store(lse3 + b * HW + p, l_all);
    Vec<VEC>::store(lse3 + plane + b * HW + p, l_bkg);
    Vec<VEC>::store(lse3 + 2 * plane + b * HW + p, l_t);
  }
  __shared__ float red[32];
  float r = block_sum(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = r;
}

// UNKD backward: d(-loss_px)/dx_c = ( p_c - [c in S_b] q0 exp(x_c - lse_b) - [1<=c<C_old] q_c ) / C_old
template <int VEC, bool ACC>
__global__ void __launch_bounds__(kStreamThreads)
unkd_bwd_kernel(const float* __restrict__ x, const float* __restrict__ t, const float* __restrict__ mask,
                float alpha, const float* __restrict__ lse3, const float* __restrict__ g_px,
                const float* __restrict__ g_scalar, float g_mul, float* __restrict__ dx, int B, int C, int Cs,
                int C_old, int mask_zero, long long HW) {
  const long long gpi = HW / VEC;
  const long long n_groups = gpi * B;
  const long long plane = (long long)B * HW;
  const float a2 = alpha * kLog2e;
  const float inv_cold = 1.f / (float)C_old;
  const float gs = (g_px == nullptr) ? g_scalar[0] * g_mul : 0.f;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups;
       g += (long long)gridDim.x * blockDim.x) {
    const long long b = g / gpi, p = (g - b * gpi) * VEC;
    const float* xp = x + (b * Cs) * HW + p;
    const float* tp = t + (b * C_old) * HW + p;
    float* dp = dx + (b * Cs) * HW + p;
    float la2[VEC], lt2[VEC], up[VEC], fb[VEC];  // fb = q0 * exp(lse_all - lse_bkg)
    {
      float la[VEC], lb[VEC], lt[VEC], gp[VEC], mk[VEC], u0[VEC];
      Vec<VEC>::load_cached(lse3 + b * HW + p, la);
      Vec<VEC>::load_cached(lse3 + plane + b * HW + p, lb);
      Vec<VEC>::load_cached(lse3 + 2 * plane + b * HW + p, lt);
      Vec<VEC>::load_cached(tp, u0);
      if (g_px != nullptr) Vec<VEC>::load_cached(g_px + b * HW + p, gp);
      if (mask != nullptr) Vec<VEC>::load_cached(mask + b * HW + p, mk);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        la2[i] = la[i] * kLog2e;
        lt2[i] = lt[i] * kLog2e;
        float u = (g_px != nullptr ? gp[i] : gs) * inv_cold;
        if (mask != nullptr) u *= mask_zero ? (mk[i] == 0.f ? 1.f : 0.f) : mk[i];
        up[i] = u;
        const float q0 = ex2f(fmaf(u0[i], a2, -lt2[i]));
        fb[i] = q0 * ex2f((la[i] - lb[i]) * kLog2e);
      }
    }
    {  // channel 0: in S_b, not an old foreground class
      float v[VEC], o[VEC];
      Vec<VEC>::load(xp, v);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float pr = ex2f(fmaf(v[i], kLog2e, -la2[i]));
        o[i] = up[i] * (pr - pr * fb[i]);
      }
      store_dx<VEC, ACC>(dp, o);
    }
#pragma unroll 4
    for (int c = 1; c < C_old; ++c) {
      float v[VEC], u[VEC], o[VEC];
      Vec<VEC>::load(xp + (long long)c * HW, v);
      Vec<VEC>::load(tp + (long long)c * HW, u);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float pr = ex2f(fmaf(v[i], kLog2e, -la2[i]));
        const float q = ex2f(fmaf(u[i], a2, -lt2[i]));
        o[i] = up[i] * (pr - q);
      }
      store_dx<VEC, ACC>(dp + (long long)c * HW, o);
    }
#pragma unroll 4
    for (int c = C_old; c < C; ++c) {
      float v[VEC], o[VEC];
      Vec<VEC>::load(xp + (long long)c * HW, v);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float pr = ex2f(fmaf(v[i], kLog2e, -la2[i]));
        o[i] = up[i] * (pr - pr * fb[i]);
      }
      store_dx<VEC, ACC>(dp + (long long)c * HW, o);
    }
    if (!ACC)
      for (int c = C; c < Cs; ++c) {  // channels outside the narrowed view get no gradient
        float o[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) o[i] = 0.f;
        Vec<VEC>::store_stream(dp + (long long)c * HW, o);
      }
  }
}

// ------------------------------------------------------------------------------------------
// UNCE + UNKD backward in ONE pass over the logits: both losses consume the same `outputs` (train.py:116,133) and both
// gradients are (upstream) x (softmax(x)_c - something): x is read once, softmax once, dx written once.  Two separate
// kernels (the second accumulating) move 2 x + t + 3 dx = 2.5 GB at the BASELINE workload, this one x + t + dx = 1.26 GB.
//   dx_c = u_ce ( p_c - [y'==0 ? [c<old_cl] p_c e^{lse - lse_old} : [c==y'] ] )           (SURVEY A.3, UNCE)
//        + u_kd ( p_c - [c in S_b] p_c q_0 e^{lse - lse_b} - [1<=c<C_old] q_c )           (UNKD; S_b = {0} U new)
// The per-pixel coefficients (pair_coef) and the per-element expression (pair_dx) are shared with the kernel that
// folds the bilinear adjoint in (unce_unkd_bwd_lowres_kernel): both form bit-identical dx.
// ------------------------------------------------------------------------------------------
struct PairArgs {
  const long long* y;
  const float *lse_all, *bkg_gap, *ce_g_px, *t, *mask, *lse3, *kd_g_px;
  long long plane;  // B * HW: stride of the lse3 planes
  float gs_ce, gs_kd, a2, inv_cold;
  int old_cl, ignore_index, C, C_old, mask_zero;
};

__device__ __forceinline__ PairArgs pair_args(const long long* y, const float* lse_all, const float* bkg_gap,
                                              const float* ce_g_px, const float* ce_g_scalar, float ce_g_mul,
                                              const float* ce_stats, int mean_over_valid, int old_cl, int ignore_index,
                                              const float* t, const float* mask, float alpha, const float* lse3,
                                              const float* kd_g_px, const float* kd_g_scalar, float kd_g_mul,
                                              int mask_zero, int B, int C, int C_old, long long HW) {
  PairArgs a;
  a.y = y, a.lse_all = lse_all, a.bkg_gap = bkg_gap, a.ce_g_px = ce_g_px, a.t = t, a.mask = mask, a.lse3 = lse3;
  a.kd_g_px = kd_g_px;
  a.plane = (long long)B * HW;
  a.a2 = alpha * kLog2e;
  a.inv_cold = 1.f / (float)C_old;
  a.gs_ce = 0.f;
  if (ce_g_px == nullptr) {
    a.gs_ce = ce_g_scalar[0] * ce_g_mul;
    if (mean_over_valid) a.gs_ce = a.gs_ce / ce_stats[1];
  }
  a.gs_kd = (kd_g_px == nullptr) ? kd_g_scalar[0] * kd_g_mul : 0.f;
  a.old_cl = old_cl, a.ignore_index = ignore_index, a.C = C, a.C_old = C_old, a.mask_zero = mask_zero;
  return a;
}

// per-pixel coefficients of VEC adjacent pixels; px = b * HW + p, tp = t + b * C_old * HW + p (its plane 0: q_0)
template <int VEC>
struct PairCoef {
  float la2[VEC], lt2[VEC], uce[VEC], ukd[VEC], fold[VEC], fb[VEC];
  int lab[VEC];
};

template <int VEC>
__device__ __forceinline__ void pair_coef(const PairArgs& a, long long px, const float* tp, PairCoef<VEC>& q) {
  float la[VEC], lo[VEC], lb[VEC], lt[VEC], gp[VEC], gk[VEC], mk[VEC], u0[VEC];
  Vec<VEC>::load_cached(a.lse_all + px, la);
  Vec<VEC>::load_cached(a.bkg_gap + px, lo);  // lse_all - lse_old where the label is 0 (the forward's loss_px)
  Vec<VEC>::load_cached(a.lse3 + a.plane + px, lb);
  Vec<VEC>::load_cached(a.lse3 + 2 * a.plane + px, lt);
  Vec<VEC>::load_cached(tp, u0);
  if (a.ce_g_px != nullptr) Vec<VEC>::load_cached(a.ce_g_px + px, gp);
  if (a.kd_g_px != nullptr) Vec<VEC>::load_cached(a.kd_g_px + px, gk);
  if (a.mask != nullptr) Vec<VEC>::load_cached(a.mask + px, mk);
  const long long* yp = a.y + px;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    long long tt = yp[i];
    if (tt < a.old_cl) tt = 0;
    const bool dead = (tt == a.ignore_index) || tt < 0 || tt >= a.C;
    q.lab[i] = dead ? -1 : (int)tt;
    q.uce[i] = dead ? 0.f : (a.ce_g_px != nullptr ? gp[i] : a.gs_ce);
    q.la2[i] = la[i] * kLog2e;
    q.lt2[i] = lt[i] * kLog2e;
    q.fold[i] = ex2f(lo[i] * kLog2e);
    float u = (a.kd_g_px != nullptr ? gk[i] : a.gs_kd) * a.inv_cold;
    if (a.mask != nullptr) u *= a.mask_zero ? (mk[i] == 0.f ? 1.f : 0.f) : mk[i];
    q.ukd[i] = u;
    const float q0 = ex2f(fmaf(u0[i], a.a2, -q.lt2[i]));
    q.fb[i] = q0 * ex2f((la[i] - lb[i]) * kLog2e);
  }
}

// dx of channel c at pixel i: v = x_c, u = t_c (read only for an old foreground class, 1 <= c < C_old)
template <int VEC>
__device__ __forceinline__ float pair_dx(const PairArgs& a, const PairCoef<VEC>& q, int i, int c, bool old_fg, float v,
                                         float u) {
  const float pr = ex2f(fmaf(v, kLog2e, -q.la2[i]));
  float sub_ce;
  if (q.lab[i] == 0 && a.old_cl > 0)
    sub_ce = (c < a.old_cl) ? pr * q.fold[i] : 0.f;
  else
    sub_ce = (c == q.lab[i]) ? 1.f : 0.f;
  const float sub_kd = old_fg ? ex2f(fmaf(u, a.a2, -q.lt2[i])) : pr * q.fb[i];
  return fmaf(q.uce[i], pr - sub_ce, q.ukd[i] * (pr - sub_kd));
}

template <int VEC, bool ACC>
__global__ void __launch_bounds__(kStreamThreads)
unce_unkd_bwd_kernel(const float* __restrict__ x, const long long* __restrict__ y, const float* __restrict__ lse_all,
                     const float* __restrict__ bkg_gap, const float* __restrict__ ce_g_px,
                     const float* __restrict__ ce_g_scalar, float ce_g_mul, const float* __restrict__ ce_stats,
                     int mean_over_valid, int old_cl, int ignore_index, const float* __restrict__ t,
                     const float* __restrict__ mask, float alpha, const float* __restrict__ lse3,
                     const float* __restrict__ kd_g_px, const float* __restrict__ kd_g_scalar, float kd_g_mul,
                     int mask_zero, float* __restrict__ dx, int B, int C, int C_old, long long HW) {
  const long long gpi = HW / VEC;
  const long long n_groups = gpi * B;
  const PairArgs a = pair_args(y, lse_all, bkg_gap, ce_g_px, ce_g_scalar, ce_g_mul, ce_stats, mean_over_valid, old_cl,
                               ignore_index, t, mask, alpha, lse3, kd_g_px, kd_g_scalar, kd_g_mul, mask_zero, B, C,
                               C_old, HW);
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups;
       g += (long long)gridDim.x * blockDim.x) {
    const long long b = g / gpi, p = (g - b * gpi) * VEC;
    const float* xp = x + (b * C) * HW + p;
    const float* tp = t + (b * C_old) * HW + p;
    float* dp = dx + (b * C) * HW + p;
    PairCoef<VEC> q;
    pair_coef<VEC>(a, b * HW + p, tp, q);
#pragma unroll 4
    for (int c = 0; c < C; ++c) {
      float v[VEC], u[VEC], o[VEC];
      Vec<VEC>::load(xp + (long long)c * HW, v);
      const bool old_fg = c >= 1 && c < C_old;  // an old foreground class: KD subtracts q_c (uniform over the block)
      if (old_fg) Vec<VEC>::load(tp + (long long)c * HW, u);
#pragma unroll
      for (int i = 0; i < VEC; ++i) o[i] = pair_dx<VEC>(a, q, i, c, old_fg, v[i], u[i]);
      store_dx<VEC, ACC>(dp + (long long)c * HW, o);
    }
  }
}

// ------------------------------------------------------------------------------------------
// The same backward contracted with the bilinear adjoint on the fly: d_lr = U^T dx with U the upsample of the logits
// (sweep form, sweep_adjoint.cuh: integer scales, a multiple of 8 along x).  dx is formed in registers and never
// written: the pass reads x, t, the labels and the saved planes once (4 C + 4 C_old + 24 B per pixel) and writes only
// the low-res gradient.
// block = (image b, range of low-res rows [y0, ylast], group of at most KMAX channels), the channel group fastest in the
// grid so that the per-pixel planes, read by every group, come from L2 after the first.  thread = 4 consecutive X of
// a full-res row (blockDim = W / 4), sweeping the full-res rows of the range top-down; per row and channel 8 FMAs fold
// x and 4 fold y into 4 accumulators: (upper, lower) y tap x (upper, lower) x tap.  When the sweep leaves interval k
// (the rows whose upper tap is k), low-res row k is emitted (shared-memory gather over the threads whose x taps hit
// each cell, fixed order) and the lower-tap sums become the next interval's starting value.  The lower-tap sums of a
// range's last interval belong to the next range's first row: that row receives exactly two contributions, its owner's
// and this carry, added with atomicAdd onto a zeroed output (two operands commute: deterministic).
// ------------------------------------------------------------------------------------------
// KMAX: channels per block (a multiple of 4); NREG: register cap per thread (blocks of <= 256 threads)
template <int KMAX, int NREG>
__global__ void __maxnreg__(NREG)
unce_unkd_bwd_lowres_kernel(const float* __restrict__ x, const long long* __restrict__ y,
                            const float* __restrict__ lse_all, const float* __restrict__ bkg_gap,
                            const float* __restrict__ ce_g_px, const float* __restrict__ ce_g_scalar, float ce_g_mul,
                            const float* __restrict__ ce_stats, int mean_over_valid, int old_cl, int ignore_index,
                            const float* __restrict__ t, const float* __restrict__ mask, float alpha,
                            const float* __restrict__ lse3, const float* __restrict__ kd_g_px,
                            const float* __restrict__ kd_g_scalar, float kd_g_mul, int mask_zero,
                            float* __restrict__ d_lr, int B, int C, int C_old, int h, int w, int H, int W,
                            float scale_h, float scale_w, int n_ranges, int range_rows, int n_cgroups, int ny_cap) {
  extern __shared__ __align__(16) uint8_t lr_dyn[];
  const int wv = blockDim.x;  // == W / 4
  const int tid = threadIdx.x;
  // 8-byte entries first: every array starts aligned whatever ny_cap and wv are
  float2* s_p = reinterpret_cast<float2*>(lr_dyn);                 // [2][KMAX][wv] (p0, p1) of the rows being emitted
  short4* s_j = reinterpret_cast<short4*>(s_p + 2 * KMAX * wv);    // [w] thread ranges hitting low-res x
  float2* s_h = reinterpret_cast<float2*>(s_j + w);                // [ny_cap] y weights (upper tap, lower tap)
  int* s_k = reinterpret_cast<int*>(s_h + ny_cap);                 // [ny_cap] low-res row of the upper tap
  int* s_x0 = s_k + ny_cap;                                        // [wv] upper / lower x tap of each thread
  int* s_x1 = s_x0 + wv;
  __shared__ int s_lim[2];
  const long long HW = (long long)H * W;
  const PairArgs a = pair_args(y, lse_all, bkg_gap, ce_g_px, ce_g_scalar, ce_g_mul, ce_stats, mean_over_valid, old_cl,
                               ignore_index, t, mask, alpha, lse3, kd_g_px, kd_g_scalar, kd_g_mul, mask_zero, B, C,
                               C_old, HW);
  const int cg = blockIdx.x % n_cgroups;
  const int rest = blockIdx.x / n_cgroups;
  const int rg = rest % n_ranges;
  const long long b = rest / n_ranges;
  const int c0 = (int)((long long)cg * C / n_cgroups), kc = (int)((long long)(cg + 1) * C / n_cgroups) - c0;
  const int y0 = rg * range_rows, ylast = min(h, y0 + range_rows) - 1;
  float wx0[4], wx1[4];
  sweep_x_taps(tid, wv, w, W, scale_w, wx0, wx1, s_x0, s_x1, s_j);
  int i_lo, i_hi;
  const int Ylo = sweep_y_taps(tid, wv, y0, ylast, h, H, scale_h, ny_cap, s_k, s_h, s_lim, i_lo, i_hi);
  const int X = tid * 4;
  const float* xb = x + (b * C + c0) * HW + X;
  const float* tb = t + b * C_old * HW + X;
  float* out = d_lr + (b * C + c0) * (long long)h * w;
  // accumulators per channel: a0 = towards low-res row `cur` (upper y tap), a1 = towards row cur + 1 (lower y tap);
  // .x / .y = upper / lower x tap
  float2 a0[KMAX], a1[KMAX];
#pragma unroll
  for (int j = 0; j < KMAX; ++j) a0[j] = a1[j] = make_float2(0.f, 0.f);
  int cur = -1, flip = 0;
  // low-res row `row` of the block's channels += gather over x of the per-thread pairs in a0; `shared`: another block
  // contributes to this row as well
  auto emit = [&](int row, bool shared) {
    float2* sp = s_p + flip * KMAX * wv;
#pragma unroll
    for (int j = 0; j < KMAX; ++j)
      if (j < kc) sp[j * wv + tid] = a0[j];
    __syncthreads();  // one barrier per emit: the buffers alternate, so the next emit cannot overtake this gather
    for (int o = tid; o < kc * w; o += wv) {
      const int j = o / w, xo = o - j * w;
      const short4 jr = s_j[xo];
      const float2* pj = sp + j * wv;
      float acc = 0.f;
      for (int i = jr.x; i < jr.y; ++i) acc += pj[i].x;
      for (int i = jr.z; i < jr.w; ++i) acc += pj[i].y;
      float* dst = out + ((long long)j * h + row) * w + xo;
      if (shared)
        atomicAdd(dst, acc);
      else
        *dst = acc;
    }
    flip ^= 1;
  };
#pragma unroll 1
  for (int i = i_lo; i < i_hi; ++i) {
    const int k = s_k[i];
    if (k != cur) {  // uniform over the block
      if (cur >= 0) {
        emit(cur, cur == y0 && y0 > 0);
#pragma unroll
        for (int j = 0; j < KMAX; ++j) a0[j] = a1[j], a1[j] = make_float2(0.f, 0.f);
      }
      cur = k;
    }
    const long long row = (long long)(Ylo + i) * W;
    PairCoef<4> q;
    pair_coef<4>(a, b * HW + row + X, tb + row, q);
    const float2 hw = s_h[i];
#pragma unroll
    for (int j0 = 0; j0 < KMAX; j0 += 4) {  // 4 channels of x and t in flight, then their arithmetic
      float v[4][4], u[4][4];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int c = c0 + j0 + jj;
        if (j0 + jj < kc) Vec<4>::load(xb + (long long)(j0 + jj) * HW + row, v[jj]);
        if (j0 + jj < kc && c >= 1 && c < C_old) Vec<4>::load(tb + (long long)c * HW + row, u[jj]);
      }
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int j = j0 + jj, c = c0 + j;
        if (j < kc) {
          const bool old_fg = c >= 1 && c < C_old;
          float o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) o[e] = pair_dx<4>(a, q, e, c, old_fg, v[jj][e], u[jj][e]);
          const float p0 = fmaf(o[3], wx0[3], fmaf(o[2], wx0[2], fmaf(o[1], wx0[1], o[0] * wx0[0])));
          const float p1 = fmaf(o[3], wx1[3], fmaf(o[2], wx1[2], fmaf(o[1], wx1[1], o[0] * wx1[0])));
          a0[j].x = fmaf(hw.x, p0, a0[j].x), a0[j].y = fmaf(hw.x, p1, a0[j].y);
          a1[j].x = fmaf(hw.y, p0, a1[j].x), a1[j].y = fmaf(hw.y, p1, a1[j].y);
        }
      }
    }
  }
  if (cur >= 0) {
    emit(cur, cur == y0 && y0 > 0);
    if (ylast < h - 1) {  // lower-tap sums of the last interval: the next range's first row
#pragma unroll
      for (int j = 0; j < KMAX; ++j) a0[j] = a1[j];
      emit(ylast + 1, true);
    }
  }
}

// MaskCrossEntropy's pixel weight (utils/loss.py:207-211): 1 where the old model predicts background
// (argmax over channels == 0; ties resolve to the first index like torch.argmax) or the label is > old_cl.
__global__ void __launch_bounds__(kStreamThreads)
bkg_mask_kernel(const float* __restrict__ t, const long long* __restrict__ y, float* __restrict__ mask, int B,
                int C_old, long long HW, int old_cl) {
  const long long n = (long long)B * HW;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += (long long)gridDim.x * blockDim.x) {
    const long long b = g / HW, p = g - b * HW;
    const float* tp = t + (b * C_old) * HW + p;
    const float t0 = ldg_stream1(tp);
    const bool t0_nan = t0 != t0;  // torch.argmax: NaN is the maximum, the first maximum wins
    bool bkg = true;
    for (int c = 1; c < C_old; ++c) {
      const float v = ldg_stream1(tp + (long long)c * HW);
      if (!t0_nan && (v > t0 || v != v)) bkg = false;
    }
    mask[g] = (bkg || y[g] > old_cl) ? 1.f : 0.f;
  }
}

static int stream_grid(long long n_groups) {
  long long blocks = (n_groups + kStreamThreads - 1) / kStreamThreads;
  if (blocks > kStreamMaxBlocks) blocks = kStreamMaxBlocks;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

static bool can_vec4(long long HW, std::initializer_list<const void*> ptrs) {
  if (HW % 4 != 0) return false;
  for (const void* p : ptrs)
    if (p != nullptr && !aligned16(p)) return false;
  return true;
}

}  // namespace ucd

using namespace ucd;

extern "C" size_t ucd_reduce_scratch_floats(void) { return (size_t)kScratchFloats; }

extern "C" int ucd_unce_fwd(const float* x, int64_t* y, float* loss_px, float* lse_all, float* lse_old,
                            float* stats, float* scratch, int B, int C, int old_cl, int64_t HW,
                            int ignore_index, void* stream) {
  UCD_CHECK_ARG(x && y && loss_px && lse_all, "ucd_unce_fwd: null pointer");
  UCD_CHECK_ARG(B > 0 && C > 0 && HW > 0, "ucd_unce_fwd: bad shape B=%d C=%d HW=%lld", B, C, (long long)HW);
  UCD_CHECK_ARG(old_cl >= 0 && old_cl <= C, "ucd_unce_fwd: old_cl=%d outside [0,%d]", old_cl, C);
  UCD_CHECK_ARG(stats == nullptr || scratch != nullptr, "ucd_unce_fwd: stats requested without scratch");
  cudaStream_t st = (cudaStream_t)stream;
  float* part = stats ? scratch : nullptr;
  const bool v4 = can_vec4(HW, {x, loss_px, lse_all, lse_old}) && aligned16(y);
  const int grid = stream_grid((long long)B * HW / (v4 ? 4 : 1));
  if (v4)
    unce_fwd_kernel<4><<<grid, kStreamThreads, 0, st>>>(x, (long long*)y, loss_px, lse_all, lse_old, part, B, C,
                                                        old_cl, HW, ignore_index);
  else
    unce_fwd_kernel<1><<<grid, kStreamThreads, 0, st>>>(x, (long long*)y, loss_px, lse_all, lse_old, part, B, C,
                                                        old_cl, HW, ignore_index);
  UCD_CHECK_LAUNCH("unce_fwd_kernel");
  if (stats) {
    reduce_partials_kernel<<<1, 256, 0, st>>>(part, grid, 2, stats, 1.f);
    UCD_CHECK_LAUNCH("reduce_partials_kernel");
  }
  return UCD_OK;
}

extern "C" int ucd_unce_bwd(const float* x, const int64_t* y, const float* lse_all, const float* bkg_gap,
                            const float* g_px, const float* g_scalar, float g_mul, const float* stats,
                            int mean_over_valid, float* dx, int accumulate, int B, int C, int old_cl, int64_t HW,
                            int ignore_index, void* stream) {
  UCD_CHECK_ARG(x && y && lse_all && bkg_gap && dx, "ucd_unce_bwd: null pointer");
  UCD_CHECK_ARG(g_px || g_scalar, "ucd_unce_bwd: need g_px or g_scalar");
  UCD_CHECK_ARG(!mean_over_valid || stats, "ucd_unce_bwd: mean_over_valid needs stats");
  UCD_CHECK_ARG(B > 0 && C > 0 && HW > 0, "ucd_unce_bwd: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  const bool v4 = can_vec4(HW, {x, lse_all, bkg_gap, g_px, dx}) && aligned16(y);
  const int grid = stream_grid((long long)B * HW / (v4 ? 4 : 1));
  auto kern = v4 ? (accumulate ? unce_bwd_kernel<4, true> : unce_bwd_kernel<4, false>)
                 : (accumulate ? unce_bwd_kernel<1, true> : unce_bwd_kernel<1, false>);
  kern<<<grid, kStreamThreads, 0, st>>>(x, (const long long*)y, lse_all, bkg_gap, g_px, g_scalar, g_mul, stats,
                                        mean_over_valid, dx, B, C, old_cl, HW, ignore_index);
  UCD_CHECK_LAUNCH("unce_bwd_kernel");
  return UCD_OK;
}

// variant 0: unbiased KD (loss.py:139-184); 1: plain KD on the first C_old channels (loss.py:112-136);
// 2: unbiased KD with the pixel weight [mask == 0] (MaskKnowledgeDistillationLoss, loss.py:218-256)
static int kd_fwd_impl(const float* x, const float* t, const float* mask, float alpha, float* out_px, float* stats,
                       float* lse3, float* scratch, int B, int C, int C_old, int64_t HW, int variant, float stats_scale,
                       void* stream) {
  UCD_CHECK_ARG(x && t && stats && lse3 && scratch, "ucd_kd_fwd: null pointer");
  UCD_CHECK_ARG(B > 0 && HW > 0 && C_old >= 1 && C >= C_old, "ucd_kd_fwd: bad shape C=%d C_old=%d", C, C_old);
  UCD_CHECK_ARG(variant >= 0 && variant <= 2, "ucd_kd_fwd: bad variant %d", variant);
  cudaStream_t st = (cudaStream_t)stream;
  const int Cu = variant == 1 ? C_old : C, mz = variant == 2 ? 1 : 0;
  const bool v4 = can_vec4(HW, {x, t, mask, out_px, lse3}) && ((long long)B * HW) % 4 == 0;
  const int grid = stream_grid((long long)B * HW / (v4 ? 4 : 1));
  if (v4)
    unkd_fwd_kernel<4><<<grid, kStreamThreads, 0, st>>>(x, t, mask, alpha, out_px, lse3, scratch, B, Cu, C, C_old, mz, HW);
  else
    unkd_fwd_kernel<1><<<grid, kStreamThreads, 0, st>>>(x, t, mask, alpha, out_px, lse3, scratch, B, Cu, C, C_old, mz, HW);
  UCD_CHECK_LAUNCH("unkd_fwd_kernel");
  reduce_partials_kernel<<<1, 256, 0, st>>>(scratch, grid, 1, stats, stats_scale);
  UCD_CHECK_LAUNCH("reduce_partials_kernel");
  return UCD_OK;
}

static int kd_bwd_impl(const float* x, const float* t, const float* mask, float alpha, const float* lse3,
                       const float* g_px, const float* g_scalar, float g_mul, float* dx, int accumulate, int B, int C,
                       int C_old, int64_t HW, int variant, void* stream) {
  UCD_CHECK_ARG(x && t && lse3 && dx, "ucd_kd_bwd: null pointer");
  UCD_CHECK_ARG(g_px || g_scalar, "ucd_kd_bwd: need g_px or g_scalar");
  UCD_CHECK_ARG(B > 0 && HW > 0 && C_old >= 1 && C >= C_old, "ucd_kd_bwd: bad shape");
  UCD_CHECK_ARG(variant >= 0 && variant <= 2, "ucd_kd_bwd: bad variant %d", variant);
  cudaStream_t st = (cudaStream_t)stream;
  const int Cu = variant == 1 ? C_old : C, mz = variant == 2 ? 1 : 0;
  const bool v4 = can_vec4(HW, {x, t, mask, g_px, lse3, dx}) && ((long long)B * HW) % 4 == 0;
  const int grid = stream_grid((long long)B * HW / (v4 ? 4 : 1));
  auto kern = v4 ? (accumulate ? unkd_bwd_kernel<4, true> : unkd_bwd_kernel<4, false>)
                 : (accumulate ? unkd_bwd_kernel<1, true> : unkd_bwd_kernel<1, false>);
  kern<<<grid, kStreamThreads, 0, st>>>(x, t, mask, alpha, lse3, g_px, g_scalar, g_mul, dx, B, Cu, C, C_old, mz, HW);
  UCD_CHECK_LAUNCH("unkd_bwd_kernel");
  return UCD_OK;
}

extern "C" int ucd_unkd_fwd(const float* x, const float* t, const float* mask, float alpha, float* out_px,
                            float* stats, float* lse3, float* scratch, int B, int C, int C_old, int64_t HW,
                            void* stream) {
  return kd_fwd_impl(x, t, mask, alpha, out_px, stats, lse3, scratch, B, C, C_old, HW, 0, 1.f, stream);
}

extern "C" int ucd_unkd_bwd(const float* x, const float* t, const float* mask, float alpha, const float* lse3,
                            const float* g_px, const float* g_scalar, float g_mul, float* dx, int accumulate, int B,
                            int C, int C_old, int64_t HW, void* stream) {
  return kd_bwd_impl(x, t, mask, alpha, lse3, g_px, g_scalar, g_mul, dx, accumulate, B, C, C_old, HW, 0, stream);
}

extern "C" int ucd_kd_fwd(const float* x, const float* t, const float* mask, float alpha, float* out_px,
                          float* stats, float* lse3, float* scratch, int B, int C, int C_old, int64_t HW,
                          int variant, float stats_scale, void* stream) {
  return kd_fwd_impl(x, t, mask, alpha, out_px, stats, lse3, scratch, B, C, C_old, HW, variant, stats_scale, stream);
}

extern "C" int ucd_kd_bwd(const float* x, const float* t, const float* mask, float alpha, const float* lse3,
                          const float* g_px, const float* g_scalar, float g_mul, float* dx, int accumulate, int B,
                          int C, int C_old, int64_t HW, int variant, void* stream) {
  return kd_bwd_impl(x, t, mask, alpha, lse3, g_px, g_scalar, g_mul, dx, accumulate, B, C, C_old, HW, variant, stream);
}

extern "C" int ucd_bkg_mask(const float* t_old, const int64_t* labels, float* mask, int B, int C_old, int64_t HW,
                            int old_cl, void* stream) {
  UCD_CHECK_ARG(t_old && labels && mask, "ucd_bkg_mask: null pointer");
  UCD_CHECK_ARG(B > 0 && C_old >= 1 && HW > 0, "ucd_bkg_mask: bad shape");
  bkg_mask_kernel<<<stream_grid((long long)B * HW), kStreamThreads, 0, (cudaStream_t)stream>>>(
      t_old, (const long long*)labels, mask, B, C_old, HW, old_cl);
  UCD_CHECK_LAUNCH("bkg_mask_kernel");
  return UCD_OK;
}

extern "C" int ucd_unce_unkd_bwd(const float* x, const int64_t* y, const float* lse_all, const float* bkg_gap,
                                 const float* ce_g_px, const float* ce_g_scalar, float ce_g_mul, const float* ce_stats,
                                 int mean_over_valid, int old_cl, int ignore_index, const float* t, const float* mask,
                                 float alpha, const float* lse3, const float* kd_g_px, const float* kd_g_scalar,
                                 float kd_g_mul, int kd_variant, float* dx, int accumulate, int B, int C, int C_old,
                                 int64_t HW, void* stream) {
  UCD_CHECK_ARG(x && y && lse_all && bkg_gap && t && lse3 && dx, "ucd_unce_unkd_bwd: null pointer");
  UCD_CHECK_ARG((ce_g_px || ce_g_scalar) && (kd_g_px || kd_g_scalar), "ucd_unce_unkd_bwd: need g_px or g_scalar for both terms");
  UCD_CHECK_ARG(!mean_over_valid || ce_stats, "ucd_unce_unkd_bwd: mean_over_valid needs stats");
  UCD_CHECK_ARG(B > 0 && HW > 0 && C_old >= 1 && C >= C_old, "ucd_unce_unkd_bwd: bad shape");
  UCD_CHECK_ARG(kd_variant == 0 || kd_variant == 2, "ucd_unce_unkd_bwd: KD variant must be 0 (unbiased) or 2 (masked)");
  cudaStream_t st = (cudaStream_t)stream;
  const bool v4 = can_vec4(HW, {x, lse_all, bkg_gap, ce_g_px, t, mask, lse3, kd_g_px, dx}) && aligned16(y) &&
                  ((long long)B * HW) % 4 == 0;
  const int grid = stream_grid((long long)B * HW / (v4 ? 4 : 1));
  auto kern = v4 ? (accumulate ? unce_unkd_bwd_kernel<4, true> : unce_unkd_bwd_kernel<4, false>)
                 : (accumulate ? unce_unkd_bwd_kernel<1, true> : unce_unkd_bwd_kernel<1, false>);
  kern<<<grid, kStreamThreads, 0, st>>>(x, (const long long*)y, lse_all, bkg_gap, ce_g_px, ce_g_scalar, ce_g_mul,
                                        ce_stats, mean_over_valid, old_cl, ignore_index, t, mask, alpha, lse3, kd_g_px,
                                        kd_g_scalar, kd_g_mul, kd_variant == 2 ? 1 : 0, dx, B, C, C_old, HW);
  UCD_CHECK_LAUNCH("unce_unkd_bwd_kernel");
  return UCD_OK;
}

extern "C" int ucd_unce_unkd_bwd_lowres(const float* x, const int64_t* y, const float* lse_all, const float* bkg_gap,
                                        const float* ce_g_px, const float* ce_g_scalar, float ce_g_mul,
                                        const float* ce_stats, int mean_over_valid, int old_cl, int ignore_index,
                                        const float* t, const float* mask, float alpha, const float* lse3,
                                        const float* kd_g_px, const float* kd_g_scalar, float kd_g_mul, int kd_variant,
                                        float* d_lr, int B, int C, int C_old, int h, int w, int H, int W,
                                        void* stream) {
  UCD_CHECK_ARG(x && y && lse_all && bkg_gap && t && lse3 && d_lr, "ucd_unce_unkd_bwd_lowres: null pointer");
  UCD_CHECK_ARG((ce_g_px || ce_g_scalar) && (kd_g_px || kd_g_scalar),
                "ucd_unce_unkd_bwd_lowres: need g_px or g_scalar for both terms");
  UCD_CHECK_ARG(!mean_over_valid || ce_stats, "ucd_unce_unkd_bwd_lowres: mean_over_valid needs stats");
  UCD_CHECK_ARG(B > 0 && C_old >= 1 && C >= C_old && h > 0 && w > 0 && H > 0 && W > 0,
                "ucd_unce_unkd_bwd_lowres: bad shape");
  UCD_CHECK_ARG(kd_variant == 0 || kd_variant == 2,
                "ucd_unce_unkd_bwd_lowres: KD variant must be 0 (unbiased) or 2 (masked)");
  // the sweep form of the adjoint (sweep_adjoint.cuh): integer scales, a multiple of 8 along x, one block row = W/4
  // threads; everything else is the caller's two-step path (ucd_unce_unkd_bwd + ucd_upsample_bilinear_bwd)
  const int up = H / h;
  const bool ok = H % h == 0 && W % w == 0 && (W / w) % 8 == 0 && W / 4 <= 256 && (W / 4) % 32 == 0 && w <= W / 4 &&
                  can_vec4((long long)H * W, {x, lse_all, bkg_gap, ce_g_px, t, mask, lse3, kd_g_px}) && aligned16(y) &&
                  up <= 64;
  if (!ok) {
    set_error("ucd_unce_unkd_bwd_lowres: %dx%d -> %dx%d is not a sweep-form shape", h, w, H, W);
    return UCD_ENOSUP;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int wv = W / 4;
  struct Variant {
    int k, nreg;
    void (*fn)(const float*, const long long*, const float*, const float*, const float*, const float*, float,
               const float*, int, int, int, const float*, const float*, float, const float*, const float*,
               const float*, float, int, float*, int, int, int, int, int, int, int, float, float, int, int, int, int);
  };
  static const Variant variants[] = {{8, 128, unce_unkd_bwd_lowres_kernel<8, 128>},
                                     {4, 128, unce_unkd_bwd_lowres_kernel<4, 128>},
#ifdef UCD_DEBUG_KNOBS  // tighter register caps: more warps per SM, a few spilled registers
                                     {4, 96, unce_unkd_bwd_lowres_kernel<4, 96>},
                                     {8, 112, unce_unkd_bwd_lowres_kernel<8, 112>},
#endif
  };
  int vi = 0;
#ifdef UCD_DEBUG_KNOBS
  if (const char* e = getenv("UCD_LRB_VARIANT")) vi = (atoi(e) >= 0 && atoi(e) < 4) ? atoi(e) : 0;  // tuning knob
#endif
  const Variant& var = variants[vi];
  // Grid: enough threads for ~2 waves of what the registers let reside per SM.  Fewer low-res rows per range first
  // (each range boundary costs one extra row emit), then more, smaller channel groups (each group re-reads the
  // per-pixel planes from L2 and recomputes the coefficients).
  const int min_groups = (C + var.k - 1) / var.k;
  int groups = min_groups, rows = h;
  const long long want = 2ll * kNumSMs * (65536 / var.nreg / 32 * 32);
  auto threads = [&](int r, int g) { return (long long)B * ((h + r - 1) / r) * g * wv; };
  while (rows > 1 && threads(rows, groups) < want) rows = (rows + 1) / 2;
  while (groups < C && threads(rows, groups) < want) ++groups;
  // the tap table of one range must fit in shared memory
  auto dyn_bytes = [&](int r) {
    return (size_t)2 * var.k * wv * 8 + (size_t)w * 8 + (size_t)((r + 2) * up + 8) * 12 + (size_t)2 * wv * 4;
  };
#ifdef UCD_DEBUG_KNOBS
  if (const char* e = getenv("UCD_LRB_ROWS")) rows = atoi(e) > 0 ? min(atoi(e), h) : rows;  // tuning knobs
  if (const char* e = getenv("UCD_LRB_GROUPS")) groups = atoi(e) >= min_groups ? min(atoi(e), C) : groups;
#endif
  while (rows > 1 && dyn_bytes(rows) > 200 * 1024) rows = (rows + 1) / 2;
  const int n_ranges = (h + rows - 1) / rows;
  const long long nb = (long long)B * n_ranges * groups;
  if (nb >= (1ll << 31) || dyn_bytes(rows) > 200 * 1024) {
    set_error("ucd_unce_unkd_bwd_lowres: B=%d h=%d H=%d needs more blocks or shared memory than one launch has", B, h, H);
    return UCD_ENOSUP;
  }
  const int ny_cap = (rows + 2) * up + 8;
  const size_t dyn = dyn_bytes(rows);
  auto kern = var.fn;
  cudaError_t e;
  if (dyn > 48 * 1024) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(unce_unkd_bwd_lowres)");
  }
  // range boundary rows receive two contributions (see the kernel): the output starts from zero
  e = cudaMemsetAsync(d_lr, 0, (size_t)B * C * h * w * sizeof(float), st);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(unce_unkd_bwd_lowres)");
  kern<<<(unsigned)nb, wv, dyn, st>>>(x, (const long long*)y, lse_all, bkg_gap, ce_g_px, ce_g_scalar, ce_g_mul,
                                      ce_stats, mean_over_valid, old_cl, ignore_index, t, mask, alpha, lse3, kd_g_px,
                                      kd_g_scalar, kd_g_mul, kd_variant == 2 ? 1 : 0, d_lr, B, C, C_old, h, w, H, W,
                                      (float)h / (float)H, (float)w / (float)W, n_ranges, rows, groups, ny_cap);
  UCD_CHECK_LAUNCH("unce_unkd_bwd_lowres_kernel");
  return UCD_OK;
}
