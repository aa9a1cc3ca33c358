// Training path of the Conv-TasNet hot path: a forward that keeps what the backward needs, and the backward itself
// (gradients of all 343 parameter tensors), i.e. what `loss.backward()` does in the reference trainer
// (egs/wsj0-mix/common/src/driver.py:146-150) for the modules of src/models/conv_tasnet.py, src/models/tdcn.py,
// src/models/filterbank.py and src/modules/norm.py.
//
// Structure (first cut: correctness and full coverage; the dense contractions already run on the tcgen05 kernels):
//   * every 1x1 convolution, forward or data-gradient (W^T dY), is ONE call of the pointwise contraction kernels of the
//     inference path (ctn_pw_umma / ctn_pw_simt, raw epilogue) -- 3xTF32 on the tensor cores by default;
//   * weight gradients dW = sum_{b,t} dY X^T reduce over B*frames (128 k at cfg2): a split-K FFMA kernel (k_wgrad,
//     64x64 register-tiled, fp32 atomics across the splits);
//   * everything between the contractions (bias, PReLU, gLN and their backward, dilated depthwise conv and its
//     backward, residual / skip bookkeeping) are streaming kernels over the (B, C, pitch) layout, HBM-bound, with the
//     per-sample gLN reductions accumulated in double.
// Saved per residual block: its input x_i, the pre-activations h_pre = W1 x + b1 and u_pre = dwconv(gLN1(PReLU h_pre)) + bd,
// and the two (sum, sumsq) statistics; normalised tensors are recomputed in the backward.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <math.h>
#include <stdlib.h>
#include "ctn_internal.h"

namespace {

struct Carver {
  char* base;
  size_t off;
  explicit Carver(void* b) : base((char*)b), off(0) {}
  template <typename T>
  T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? (T*)(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

// ================================================================================================================
// streaming kernels.  Layout (B, C, pitch), pitch % 128 == 0, rows 16-byte aligned; only columns t < frames carry data,
// pad columns are written as zero.  A thread owns 4 consecutive time steps (128-bit loads / stores).
// Unless noted: grid (min(C, 1024), B), block 256, a block walks channels c = blockIdx.x, += gridDim.x.
// ================================================================================================================
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
// zero the lanes of a 4-vector that fall at or beyond `frames`
__device__ __forceinline__ float4 mask4(float4 v, int t, int frames) {
  if (t + 3 < frames) return v;
  if (t + 0 >= frames) v.x = 0.f;
  if (t + 1 >= frames) v.y = 0.f;
  if (t + 2 >= frames) v.z = 0.f;
  if (t + 3 >= frames) v.w = 0.f;
  return v;
}
// 4 consecutive samples row[t0 .. t0+3] with zero outside [0, frames) (any alignment, any t0)
__device__ __forceinline__ float4 ld4_shift(const float* __restrict__ row, int t0, int frames) {
  if ((t0 & 3) == 0 && t0 >= 0 && t0 + 3 < frames) return ld4(row + t0);
  float4 v;
  v.x = (t0 + 0 >= 0 && t0 + 0 < frames) ? row[t0 + 0] : 0.f;
  v.y = (t0 + 1 >= 0 && t0 + 1 < frames) ? row[t0 + 1] : 0.f;
  v.z = (t0 + 2 >= 0 && t0 + 2 < frames) ? row[t0 + 2] : 0.f;
  v.w = (t0 + 3 >= 0 && t0 + 3 < frames) ? row[t0 + 3] : 0.f;
  return v;
}
__device__ __forceinline__ float4 prelu4(float4 v, float a) {
  return make_float4(prelu_f(v.x, a), prelu_f(v.y, a), prelu_f(v.z, a), prelu_f(v.w, a));
}
__device__ __forceinline__ float sum4(float4 v) { return (v.x + v.y) + (v.z + v.w); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w))); }

// y = y + bias[c] (in place) ; stats[b] += (sum, sumsq) of PReLU(y)          (tdcn.py:116-119 before the norm)
__global__ void __launch_bounds__(256) k_bias_prelu_stats(float* __restrict__ y, const float* __restrict__ bias,
                                                          const float* __restrict__ slope, double* __restrict__ stats, int C,
                                                          int frames, int pitch) {
  __shared__ double red[64];
  const int b = blockIdx.y;
  const float a = slope[0];
  double s = 0.0, ss = 0.0;
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    float* r = y + ((size_t)b * C + c) * pitch;
    const float bc = bias[c];
    float ls = 0.f, lss = 0.f;
    for (int t = threadIdx.x * 4; t < pitch; t += 1024) {
      float4 v = zero4();
      if (t < frames) {
        v = ld4(r + t);
        v = mask4(make_float4(v.x + bc, v.y + bc, v.z + bc, v.w + bc), t, frames);
        const float4 p = prelu4(v, a);
        ls += sum4(p);
        lss += dot4(p, p);
      }
      st4(r + t, v);
    }
    s += ls;
    ss += lss;
  }
  block_sum2_d(s, ss, red);
  if (threadIdx.x == 0) { atomicAdd(&stats[2 * b], s); atomicAdd(&stats[2 * b + 1], ss); }
}

// u_pre[c][t] = sum_k wd[c][k] * hn[c][t + k*d - pl] + bd[c],  hn = gLN1(PReLU(h_pre)) inside [0,frames), 0 outside
// (tdcn.py:120-130,181); stats2[b] += (sum, sumsq) of PReLU(u_pre; a2)
#define CTN_MAX_P 8
__global__ void __launch_bounds__(256) k_dw_train_fwd(const float* __restrict__ hpre, float* __restrict__ upre,
                                                      const float* __restrict__ g1, const float* __restrict__ b1,
                                                      const float* __restrict__ wd, const float* __restrict__ bd,
                                                      const float* __restrict__ slope1, const float* __restrict__ slope2,
                                                      const double* __restrict__ stats1, double* __restrict__ stats2, int C,
                                                      int frames, int pitch, int P, int dil, int pad_left, double n1, float eps) {
  __shared__ double red[64];
  const int b = blockIdx.y;
  const float a1 = slope1[0], a2 = slope2[0];
  const float2 mr = gln_mean_rstd(stats1 + 2 * b, n1, eps);
  double s = 0.0, ss = 0.0;
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    const float* h = hpre + ((size_t)b * C + c) * pitch;
    float* u = upre + ((size_t)b * C + c) * pitch;
    const float gsc = g1[c] * mr.y, gsh = b1[c] - mr.x * mr.y * g1[c];
    const float bc = bd[c];
    float ls = 0.f, lss = 0.f;
    for (int t = threadIdx.x * 4; t < pitch; t += 1024) {
      float4 v = zero4();
      if (t < frames) {
        v = make_float4(bc, bc, bc, bc);
        for (int k = 0; k < P; ++k) {
          const int t0 = t + k * dil - pad_left;
          const float w = wd[c * P + k];
          const float4 q = prelu4(ld4_shift(h, t0, frames), a1);
          // hn = gsc*q + gsh inside [0,frames), exactly 0 outside (the zero padding is applied AFTER the norm, tdcn.py:123-130)
          if (t0 + 0 >= 0 && t0 + 0 < frames) v.x = fmaf(w, fmaf(gsc, q.x, gsh), v.x);
          if (t0 + 1 >= 0 && t0 + 1 < frames) v.y = fmaf(w, fmaf(gsc, q.y, gsh), v.y);
          if (t0 + 2 >= 0 && t0 + 2 < frames) v.z = fmaf(w, fmaf(gsc, q.z, gsh), v.z);
          if (t0 + 3 >= 0 && t0 + 3 < frames) v.w = fmaf(w, fmaf(gsc, q.w, gsh), v.w);
        }
        v = mask4(v, t, frames);
        const float4 p = mask4(prelu4(v, a2), t, frames);
        ls += sum4(p);
        lss += dot4(p, p);
      }
      st4(u + t, v);
    }
    s += ls;
    ss += lss;
  }
  block_sum2_d(s, ss, red);
  if (threadIdx.x == 0) { atomicAdd(&stats2[2 * b], s); atomicAdd(&stats2[2 * b + 1], ss); }
}

// y = gLN(act(pre)) : act = PReLU(slope) or identity (slope == nullptr)
__global__ void __launch_bounds__(256) k_act_norm(const float* __restrict__ pre, float* __restrict__ y,
                                                  const float* __restrict__ slope, const float* __restrict__ g,
                                                  const float* __restrict__ bt, const double* __restrict__ stats, double n,
                                                  float eps, int C, int frames, int pitch) {
  const int b = blockIdx.y;
  const float2 mr = gln_mean_rstd(stats + 2 * b, n, eps);
  const bool act = slope != nullptr;
  const float a = act ? slope[0] : 1.f;
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    const float* p = pre + ((size_t)b * C + c) * pitch;
    float* o = y + ((size_t)b * C + c) * pitch;
    const float gsc = g[c] * mr.y, gsh = bt[c] - mr.x * mr.y * g[c];
    // 4 independent 128-bit loads in flight per thread before any of them is used (memory-level parallelism)
    for (int tb = threadIdx.x * 4; tb < pitch; tb += 4096) {
      float4 x[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = tb + u * 1024;
        x[u] = t < frames ? ld4(p + t) : zero4();
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = tb + u * 1024;
        if (t >= pitch) break;
        float4 v = zero4();
        if (t < frames) {
          float4 q = x[u];
          if (act) q = prelu4(q, a);
          v = mask4(make_float4(fmaf(gsc, q.x, gsh), fmaf(gsc, q.y, gsh), fmaf(gsc, q.z, gsh), fmaf(gsc, q.w, gsh)), t, frames);
        }
        st4(o + t, v);
      }
    }
  }
}

// rows of r (B, Mt, pitch): m < Bc (has_out): x_out = x_in + r + bo[m] ; else skip (+)= r + bs[j]      (tdcn.py:144-145, :39)
__global__ void __launch_bounds__(256) k_res_skip(const float* __restrict__ r, int Mt, const float* __restrict__ xin,
                                                  float* __restrict__ xout, float* __restrict__ skip,
                                                  const float* __restrict__ bo, const float* __restrict__ bs, int Bc, int Sc,
                                                  int has_out, int skip_init, int frames, int pitch) {
  const int b = blockIdx.y;
  for (int m = blockIdx.x; m < Mt; m += gridDim.x) {
    const float* rr = r + ((size_t)b * Mt + m) * pitch;
    const bool is_x = has_out && m < Bc;
    const int j = m - (has_out ? Bc : 0);
    const float* src = is_x ? xin + ((size_t)b * Bc + m) * pitch : skip + ((size_t)b * Sc + j) * pitch;
    float* dst = is_x ? xout + ((size_t)b * Bc + m) * pitch : skip + ((size_t)b * Sc + j) * pitch;
    const float bb = is_x ? bo[m] : bs[j];
    const bool fresh = !is_x && skip_init;
    for (int t = threadIdx.x * 4; t < pitch; t += 1024) {
      float4 v = zero4();
      if (t < frames) {
        const float4 q = ld4(rr + t);
        const float4 base = fresh ? zero4() : ld4(src + t);
        v = mask4(make_float4(base.x + q.x + bb, base.y + q.y + bb, base.z + q.z + bb, base.w + q.w + bb), t, frames);
      }
      st4(dst + t, v);
    }
  }
}

__global__ void __launch_bounds__(256) k_transpose(const float* __restrict__ W, float* __restrict__ Wt, int M, int K) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < M * K) {
    const int m = i / K, k = i - m * K;
    Wt[(size_t)k * M + m] = W[i];
  }
}

// dst[b][c][:] (+)= src[b][c][:] for c < C, with independent batch strides (row blocks of wider tensors)
__global__ void __launch_bounds__(256) k_rows(float* __restrict__ dst, size_t dst_bs, const float* __restrict__ src,
                                              size_t src_bs, int C, int accumulate, int frames, int pitch) {
  const int b = blockIdx.y;
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    float* d = dst + (size_t)b * dst_bs + (size_t)c * pitch;
    const float* s = src + (size_t)b * src_bs + (size_t)c * pitch;
    for (int t = threadIdx.x * 4; t < pitch; t += 1024) {
      float4 v = zero4();
      if (t < frames) {
        v = ld4(s + t);
        if (accumulate) { const float4 q = ld4(d + t); v = make_float4(v.x + q.x, v.y + q.y, v.z + q.z, v.w + q.w); }
        v = mask4(v, t, frames);
      }
      st4(d + t, v);
    }
  }
}

// out[c] += sum_{b,t} dy[b][c][t]   (bias gradients).  grid (C, B), block 256
__global__ void __launch_bounds__(256) k_rowsum(const float* __restrict__ dy, size_t batch_stride, int frames, int pitch,
                                                float* __restrict__ out) {
  __shared__ double red[64];
  const int c = blockIdx.x, b = blockIdx.y;
  const float* r = dy + (size_t)b * batch_stride + (size_t)c * pitch;
  float ls = 0.f;
  for (int t = threadIdx.x * 4; t < frames; t += 1024) ls += sum4(mask4(ld4(r + t), t, frames));
  double s = ls, z = 0.0;
  block_sum2_d(s, z, red);
  if (threadIdx.x == 0) atomicAdd(&out[c], (float)s);
}

// ---- gLN backward, phase 1.  xhat = (act(pre) - mean) * rstd, g = gamma_c * dy:
//   sums[b] += (sum g, sum g*xhat) ; dgamma[c] += sum dy*xhat ; dbeta[c] += sum dy         grid (C, B)
__global__ void __launch_bounds__(256) k_gln_bwd_reduce(const float* __restrict__ dy, const float* __restrict__ pre,
                                                        const float* __restrict__ slope, const float* __restrict__ g,
                                                        const double* __restrict__ stats, double n, float eps,
                                                        double* __restrict__ sums, float* __restrict__ dgamma,
                                                        float* __restrict__ dbeta, int C, int frames, int pitch) {
  __shared__ double red[64];
  const int c = blockIdx.x, b = blockIdx.y;
  const float2 mr = gln_mean_rstd(stats + 2 * b, n, eps);
  const bool act = slope != nullptr;
  const float a = act ? slope[0] : 1.f;
  const float* d = dy + ((size_t)b * C + c) * pitch;
  const float* p = pre + ((size_t)b * C + c) * pitch;
  float s0 = 0.f, s1 = 0.f;
  for (int tb = threadIdx.x * 4; tb < frames; tb += 4096) {
    float4 dq[4], xq[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = tb + u * 1024;
      dq[u] = t < frames ? ld4(d + t) : zero4();
      xq[u] = t < frames ? ld4(p + t) : zero4();
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = tb + u * 1024;
      if (t < frames) {
        const float4 dv = mask4(dq[u], t, frames);
        float4 x = xq[u];
        if (act) x = prelu4(x, a);
        const float4 xh = make_float4((x.x - mr.x) * mr.y, (x.y - mr.x) * mr.y, (x.z - mr.x) * mr.y, (x.w - mr.x) * mr.y);
        s0 += sum4(dv);
        s1 += dot4(dv, xh);  // dv is zero in the pad lanes
      }
    }
  }
  double ds0 = s0, ds1 = s1;
  block_sum2_d(ds0, ds1, red);
  if (threadIdx.x == 0) {
    atomicAdd(&dbeta[c], (float)ds0);
    atomicAdd(&dgamma[c], (float)ds1);
    const double gc = (double)g[c];
    atomicAdd(&sums[2 * b], gc * ds0);
    atomicAdd(&sums[2 * b + 1], gc * ds1);
  }
}

// ---- gLN backward, phase 2 (+ the PReLU in front of the norm, + the bias of the conv that produced `pre`):
//   d_act = rstd * (g - mean(g) - xhat * mean(g*xhat))                       (GroupNorm(1,C) backward)
//   d_pre = d_act * (pre > 0 ? 1 : a) ; dslope += sum_{pre<=0} d_act * pre   (PReLU backward, single shared slope)
//   dbias[c] += sum d_pre.   dpre may alias dy.                               grid (C, B)
__global__ void __launch_bounds__(256) k_gln_prelu_bwd_apply(const float* dy, const float* __restrict__ pre, float* dpre,
                                                             const float* __restrict__ slope, const float* __restrict__ g,
                                                             const double* __restrict__ stats, double n, float eps,
                                                             const double* __restrict__ sums, float* __restrict__ dslope,
                                                             float* __restrict__ dbias, int C, int frames, int pitch) {
  __shared__ double red[64];
  const int c = blockIdx.x, b = blockIdx.y;
  const float2 mr = gln_mean_rstd(stats + 2 * b, n, eps);
  const float mg = (float)(sums[2 * b] / n), mgx = (float)(sums[2 * b + 1] / n);
  const bool act = slope != nullptr;
  const float a = act ? slope[0] : 1.f;
  const float gc = g[c];
  const float* d = dy + ((size_t)b * C + c) * pitch;
  const float* p = pre + ((size_t)b * C + c) * pitch;
  float* o = dpre + ((size_t)b * C + c) * pitch;
  float sa = 0.f, sb = 0.f;
  for (int tb = threadIdx.x * 4; tb < pitch; tb += 4096) {
   float4 dq[4], pq[4];
#pragma unroll
   for (int u = 0; u < 4; ++u) {  // all loads of the batch before the first (possibly aliasing, in-place) store
     const int t = tb + u * 1024;
     dq[u] = t < frames ? ld4(d + t) : zero4();
     pq[u] = t < frames ? ld4(p + t) : zero4();
   }
#pragma unroll
   for (int u = 0; u < 4; ++u) {
    const int t = tb + u * 1024;
    if (t >= pitch) break;
    float4 v = zero4();
    if (t < frames) {
      const float4 dv = dq[u], pv = pq[u];
      const float dvv[4] = {dv.x, dv.y, dv.z, dv.w}, pvv[4] = {pv.x, pv.y, pv.z, pv.w};
      float ov[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float x = act ? prelu_f(pvv[j], a) : pvv[j];
        const float xh = (x - mr.x) * mr.y;
        const float da = mr.y * (gc * dvv[j] - mg - xh * mgx);
        float r = da;
        if (act) {
          r = pvv[j] > 0.f ? da : a * da;
          if (!(pvv[j] > 0.f) && t + j < frames) sa = fmaf(da, pvv[j], sa);
        }
        ov[j] = t + j < frames ? r : 0.f;
        sb += ov[j];
      }
      v = make_float4(ov[0], ov[1], ov[2], ov[3]);
    }
    st4(o + t, v);
   }
  }
  double dsa = sa, dsb = sb;
  block_sum2_d(dsa, dsb, red);
  if (threadIdx.x == 0) {
    if (act && dslope) atomicAdd(dslope, (float)dsa);
    if (dbias) atomicAdd(&dbias[c], (float)dsb);
  }
}

// ---- depthwise conv backward (tdcn.py:181 with the padding of :123-130).  dU = d_u_pre (zero outside [0,frames)):
//   d_hn[c][t] = sum_k wd[c][k] * dU[c][t - k*d + pl]
//   dwd[c][k] += sum_{b,t} dU[c][t] * hn[c][t + k*d - pl],   hn = gLN1(PReLU(h_pre)) inside [0,frames), 0 outside
// grid (C, B)
__global__ void __launch_bounds__(256) k_dw_bwd(const float* __restrict__ dupre, const float* __restrict__ hpre,
                                                float* __restrict__ dhn, const float* __restrict__ slope1,
                                                const float* __restrict__ g1, const float* __restrict__ b1,
                                                const double* __restrict__ stats1, double n1, float eps,
                                                const float* __restrict__ wd, float* __restrict__ dwd,
                                                double* __restrict__ sums, float* __restrict__ dgamma,
                                                float* __restrict__ dbeta, int C, int frames, int pitch, int P, int dil,
                                                int pad_left) {
  const int c = blockIdx.x, b = blockIdx.y;
  const float a1 = slope1[0];
  const float2 mr = gln_mean_rstd(stats1 + 2 * b, n1, eps);
  const float gsc = g1[c] * mr.y, gsh = b1[c] - mr.x * mr.y * g1[c];
  float s0 = 0.f, s1 = 0.f;  // phase 1 of the gLN1 backward on the d_hn this kernel produces (saves a pass over d_hn and h)
  const float* du = dupre + ((size_t)b * C + c) * pitch;
  const float* h = hpre + ((size_t)b * C + c) * pitch;
  float* o = dhn + ((size_t)b * C + c) * pitch;
  float w[CTN_MAX_P], acc[CTN_MAX_P];
#pragma unroll
  for (int k = 0; k < CTN_MAX_P; ++k) { w[k] = k < P ? wd[c * P + k] : 0.f; acc[k] = 0.f; }
  for (int t = threadIdx.x * 4; t < pitch; t += 1024) {
    float4 v = zero4();
    if (t < frames) {
      const float4 dut = mask4(ld4(du + t), t, frames);
#pragma unroll
      for (int k = 0; k < CTN_MAX_P; ++k) {
        if (k < P) {
          const float4 q = ld4_shift(du, t - k * dil + pad_left, frames);  // u[ts] read hn[t] through tap k
          v.x = fmaf(w[k], q.x, v.x); v.y = fmaf(w[k], q.y, v.y); v.z = fmaf(w[k], q.z, v.z); v.w = fmaf(w[k], q.w, v.w);
          const int th = t + k * dil - pad_left;                           // u[t] read hn[th] through tap k
          const float4 hq = prelu4(ld4_shift(h, th, frames), a1);
          float4 hn;
          hn.x = (th + 0 >= 0 && th + 0 < frames) ? fmaf(gsc, hq.x, gsh) : 0.f;
          hn.y = (th + 1 >= 0 && th + 1 < frames) ? fmaf(gsc, hq.y, gsh) : 0.f;
          hn.z = (th + 2 >= 0 && th + 2 < frames) ? fmaf(gsc, hq.z, gsh) : 0.f;
          hn.w = (th + 3 >= 0 && th + 3 < frames) ? fmaf(gsc, hq.w, gsh) : 0.f;
          acc[k] += dot4(dut, hn);
        }
      }
      v = mask4(v, t, frames);
      const float4 hc = prelu4(ld4(h + t), a1);
      const float4 xh = make_float4((hc.x - mr.x) * mr.y, (hc.y - mr.x) * mr.y, (hc.z - mr.x) * mr.y, (hc.w - mr.x) * mr.y);
      s0 += sum4(v);
      s1 += dot4(v, xh);  // v is zero in the pad lanes
    }
    st4(o + t, v);
  }
  // one block-wide reduction for all per-row sums: P tap gradients + the two gLN1 sums (warp shuffles, then 8 partials each)
  {
    __shared__ float part[8][CTN_MAX_P + 2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < CTN_MAX_P; ++k) {
      if (k < P) {
        const float v = warp_sum(acc[k]);
        if (lane == 0) part[wid][k] = v;
      }
    }
    const float v0 = warp_sum(s0), v1 = warp_sum(s1);
    if (lane == 0) { part[wid][CTN_MAX_P] = v0; part[wid][CTN_MAX_P + 1] = v1; }
    __syncthreads();
    if (threadIdx.x < CTN_MAX_P + 2) {
      const int k = threadIdx.x;
      if (k < P || k >= CTN_MAX_P) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += (double)part[w][k];
        if (k < P) atomicAdd(&dwd[c * P + k], (float)t);
        else if (k == CTN_MAX_P) { atomicAdd(&dbeta[c], (float)t); atomicAdd(&sums[2 * b], (double)g1[c] * t); }
        else { atomicAdd(&dgamma[c], (float)t); atomicAdd(&sums[2 * b + 1], (double)g1[c] * t); }
      }
    }
  }
}

// ---- mask head backward (conv_tasnet.py:158-160 and the sigmoid of :375):  w_hat[s] = w * mask[s]
//   d_wprod[b][n][t] = sum_s d_what[b][s][n][t] * mask[b][s][n][t]
//   d_mpre = d_what * w * mask * (1 - mask)      (in place over d_what)                      grid (N, B)
__global__ void __launch_bounds__(256) k_mask_bwd(float* __restrict__ dwhat, const float* __restrict__ w,
                                                  const float* __restrict__ mask, float* __restrict__ dwprod, int S, int N,
                                                  int frames, int pitch) {
  const int b = blockIdx.y;
  for (int n = blockIdx.x; n < N; n += gridDim.x) {
    const float* wr = w + ((size_t)b * N + n) * pitch;
    float* dp = dwprod + ((size_t)b * N + n) * pitch;
    for (int t = threadIdx.x * 4; t < pitch; t += 1024) {
      float4 acc = zero4();
      const float4 wv = t < frames ? mask4(ld4(wr + t), t, frames) : zero4();
      for (int s = 0; s < S; ++s) {
        const size_t idx = (((size_t)b * S + s) * N + n) * pitch + t;
        float4 v = zero4();
        if (t < frames) {
          const float4 d = mask4(ld4(dwhat + idx), t, frames), m = ld4(mask + idx);
          acc.x = fmaf(d.x, m.x, acc.x); acc.y = fmaf(d.y, m.y, acc.y); acc.z = fmaf(d.z, m.z, acc.z); acc.w = fmaf(d.w, m.w, acc.w);
          v = make_float4(d.x * wv.x * m.x * (1.f - m.x), d.y * wv.y * m.y * (1.f - m.y), d.z * wv.z * m.z * (1.f - m.z),
                          d.w * wv.w * m.w * (1.f - m.w));
        }
        st4(dwhat + idx, v);
      }
      st4(dp + t, acc);
    }
  }
}

__global__ void __launch_bounds__(256) k_prelu_apply(const float* __restrict__ x, float* __restrict__ y,
                                                     const float* __restrict__ slope, int C, int frames, int pitch) {
  const int b = blockIdx.y;
  const float a = slope[0];
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    const float* p = x + ((size_t)b * C + c) * pitch;
    float* o = y + ((size_t)b * C + c) * pitch;
    for (int t = threadIdx.x * 4; t < pitch; t += 1024) st4(o + t, t < frames ? mask4(prelu4(ld4(p + t), a), t, frames) : zero4());
  }
}

// d_pre = dy * (pre > 0 ? 1 : a) ; dslope += sum_{pre<=0} dy*pre.  dpre may alias dy.  grid (C, B)
__global__ void __launch_bounds__(256) k_prelu_bwd(const float* dy, const float* __restrict__ pre, float* dpre,
                                                   const float* __restrict__ slope, float* __restrict__ dslope, int C,
                                                   int frames, int pitch) {
  __shared__ double red[64];
  const int c = blockIdx.x, b = blockIdx.y;
  const float a = slope[0];
  const float* d = dy + ((size_t)b * C + c) * pitch;
  const float* p = pre + ((size_t)b * C + c) * pitch;
  float* o = dpre + ((size_t)b * C + c) * pitch;
  float sa = 0.f;
  for (int t = threadIdx.x; t < pitch; t += 256) {
    float v = 0.f;
    if (t < frames) {
      const float pv = p[t], dv = d[t];
      v = pv > 0.f ? dv : a * dv;
      if (!(pv > 0.f)) sa = fmaf(dv, pv, sa);
    }
    o[t] = v;
  }
  double dsa = sa, z = 0.0;
  block_sum2_d(dsa, z, red);
  if (threadIdx.x == 0) atomicAdd(dslope, (float)dsa);
}

// d_w = d_wnorm + d_wprod, times (w > 0) when the encoder has a ReLU (filterbank.py:225-226)
__global__ void __launch_bounds__(256) k_dw_combine(float* __restrict__ dw, const float* __restrict__ dwprod,
                                                    const float* __restrict__ w, int relu, int C, int frames, int pitch) {
  const int b = blockIdx.y;
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    const size_t base = ((size_t)b * C + c) * pitch;
    for (int t = threadIdx.x; t < pitch; t += 256) {
      float v = 0.f;
      if (t < frames) {
        v = dw[base + t] + dwprod[base + t];
        if (relu && !(w[base + t] > 0.f)) v = 0.f;
      }
      dw[base + t] = v;
    }
  }
}

// ---- filter-bank weight gradients: dW[n][k] += sum_{r,f} act[r][n][f] * sig[r][f*stride + k - pl]
// (encoder: act = d_w, sig = mixture, filterbank.py:212,222; decoder: act = w_hat, sig = d_out, filterbank.py:243).
// Fast variant (L <= 32): grid (N, row groups), block 256; a thread walks frames of its rows with all L taps in registers
// (the signal window comes from L1: neighbouring frames share L - stride samples), one reduction per block at the end.
#define ENCDEC_MAX_L 32
__global__ void __launch_bounds__(256) k_encdec_wgrad(const float* __restrict__ act, const float* __restrict__ sig,
                                                      float* __restrict__ dW, int R, int N, int frames, int pitch, int T, int L,
                                                      int stride, int pad_left) {
  __shared__ float sacc[ENCDEC_MAX_L];
  const int n = blockIdx.x;
  float acc[ENCDEC_MAX_L];
#pragma unroll
  for (int k = 0; k < ENCDEC_MAX_L; ++k) acc[k] = 0.f;
  if (threadIdx.x < ENCDEC_MAX_L) sacc[threadIdx.x] = 0.f;
  __syncthreads();
  const bool vec = (L % 4 == 0) && (stride % 4 == 0) && (pad_left % 4 == 0) && (T % 4 == 0) && ((((uintptr_t)sig) & 15) == 0);
  for (int r = blockIdx.y; r < R; r += gridDim.y) {
    const float* a = act + ((size_t)r * N + n) * pitch;
    const float* sg = sig + (size_t)r * T;
    for (int f = threadIdx.x; f < frames; f += 256) {
      const float av = a[f];
      const int t0 = f * stride - pad_left;
      if (t0 >= 0 && t0 + L <= T && vec) {
        // 128-bit loads of the window (a warp's windows are 4*stride bytes apart: 4x fewer L1 wavefronts than scalar)
#pragma unroll
        for (int k4 = 0; k4 < ENCDEC_MAX_L / 4; ++k4) {
          if (k4 * 4 < L) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(sg + t0) + k4);
            acc[k4 * 4 + 0] = fmaf(av, q.x, acc[k4 * 4 + 0]);
            acc[k4 * 4 + 1] = fmaf(av, q.y, acc[k4 * 4 + 1]);
            acc[k4 * 4 + 2] = fmaf(av, q.z, acc[k4 * 4 + 2]);
            acc[k4 * 4 + 3] = fmaf(av, q.w, acc[k4 * 4 + 3]);
          }
        }
      } else if (t0 >= 0 && t0 + L <= T) {
#pragma unroll
        for (int k = 0; k < ENCDEC_MAX_L; ++k)
          if (k < L) acc[k] = fmaf(av, sg[t0 + k], acc[k]);
      } else {
#pragma unroll
        for (int k = 0; k < ENCDEC_MAX_L; ++k)
          if (k < L && t0 + k >= 0 && t0 + k < T) acc[k] = fmaf(av, sg[t0 + k], acc[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < ENCDEC_MAX_L; ++k) {
    if (k < L) {
      const float v = warp_sum(acc[k]);
      if ((threadIdx.x & 31) == 0) atomicAdd(&sacc[k], v);
    }
  }
  __syncthreads();
  if (threadIdx.x < L) atomicAdd(&dW[n * L + threadIdx.x], sacc[threadIdx.x]);
}
// generic variant (any L): grid (L, N), block 256
__global__ void __launch_bounds__(256) k_encdec_wgrad_generic(const float* __restrict__ act, const float* __restrict__ sig,
                                                              float* __restrict__ dW, int R, int N, int frames, int pitch, int T,
                                                              int L, int stride, int pad_left) {
  __shared__ double red[64];
  const int k = blockIdx.x, n = blockIdx.y;
  double s = 0.0, z = 0.0;
  for (int r = 0; r < R; ++r) {
    const float* a = act + ((size_t)r * N + n) * pitch;
    const float* sg = sig + (size_t)r * T;
    float ls = 0.f;
    for (int f = threadIdx.x; f < frames; f += 256) {
      const int t = f * stride + k - pad_left;
      if (t >= 0 && t < T) ls = fmaf(a[f], sg[t], ls);
    }
    s += ls;
  }
  block_sum2_d(s, z, red);
  if (threadIdx.x == 0) atomicAdd(&dW[n * L + k], (float)s);
}

// ---- weight gradient of a 1x1 conv: dW[m][k] += sum_{b, t<frames} dY[b][m][t] * X[b][k][t]
// 64x64 output tile per CTA, 256 threads x (4x4) accumulators, time in chunks of 32 staged TRANSPOSED in shared memory so
// that the inner product reads two conflict-free 128-bit vectors per step; grid (tiles_m*tiles_k, splits): each CTA
// reduces its share of the B*ceil(frames/32) chunks and adds its partial tile with fp32 atomics.
#define WG_T 32
__global__ void __launch_bounds__(256) k_wgrad(const float* __restrict__ dy, size_t dy_bs, const float* __restrict__ x,
                                               size_t x_bs, float* __restrict__ dW, int M, int K, int B, int frames, int pitch,
                                               int units_per_cta) {
  __shared__ __align__(16) float sdy[WG_T][68];
  __shared__ __align__(16) float sx[WG_T][68];
  const int tiles_k = (K + 63) / 64;
  const int m0 = ((int)blockIdx.x / tiles_k) * 64, k0 = ((int)blockIdx.x % tiles_k) * 64;
  const int chunks = (frames + WG_T - 1) / WG_T;
  const long long total = (long long)B * chunks;
  const long long u0 = (long long)blockIdx.y * units_per_cta;
  const long long u1 = u0 + units_per_cta < total ? u0 + units_per_cta : total;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lrow = threadIdx.x >> 2, lt = (threadIdx.x & 3) * 8;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (long long u = u0; u < u1; ++u) {
    const int b = (int)(u / chunks), t0 = (int)(u % chunks) * WG_T;
    float vy[8], vx[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { vy[j] = 0.f; vx[j] = 0.f; }
    if (m0 + lrow < M) {
      const float4* p = reinterpret_cast<const float4*>(dy + (size_t)b * dy_bs + (size_t)(m0 + lrow) * pitch + t0 + lt);
      const float4 q0 = __ldg(p), q1 = __ldg(p + 1);
      vy[0] = q0.x; vy[1] = q0.y; vy[2] = q0.z; vy[3] = q0.w; vy[4] = q1.x; vy[5] = q1.y; vy[6] = q1.z; vy[7] = q1.w;
    }
    if (k0 + lrow < K) {
      const float4* p = reinterpret_cast<const float4*>(x + (size_t)b * x_bs + (size_t)(k0 + lrow) * pitch + t0 + lt);
      const float4 q0 = __ldg(p), q1 = __ldg(p + 1);
      vx[0] = q0.x; vx[1] = q0.y; vx[2] = q0.z; vx[3] = q0.w; vx[4] = q1.x; vx[5] = q1.y; vx[6] = q1.z; vx[7] = q1.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const bool ok = t0 + lt + j < frames;  // pad columns never contribute
      sdy[lt + j][lrow] = ok ? vy[j] : 0.f;
      sx[lt + j][lrow] = ok ? vx[j] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int tt = 0; tt < WG_T; ++tt) {
      const float4 a = *reinterpret_cast<const float4*>(&sdy[tt][ty * 4]);
      const float4 c = *reinterpret_cast<const float4*>(&sx[tt][tx * 4]);
      acc[0][0] = fmaf(a.x, c.x, acc[0][0]); acc[0][1] = fmaf(a.x, c.y, acc[0][1]);
      acc[0][2] = fmaf(a.x, c.z, acc[0][2]); acc[0][3] = fmaf(a.x, c.w, acc[0][3]);
      acc[1][0] = fmaf(a.y, c.x, acc[1][0]); acc[1][1] = fmaf(a.y, c.y, acc[1][1]);
      acc[1][2] = fmaf(a.y, c.z, acc[1][2]); acc[1][3] = fmaf(a.y, c.w, acc[1][3]);
      acc[2][0] = fmaf(a.z, c.x, acc[2][0]); acc[2][1] = fmaf(a.z, c.y, acc[2][1]);
      acc[2][2] = fmaf(a.z, c.z, acc[2][2]); acc[2][3] = fmaf(a.z, c.w, acc[2][3]);
      acc[3][0] = fmaf(a.w, c.x, acc[3][0]); acc[3][1] = fmaf(a.w, c.y, acc[3][1]);
      acc[3][2] = fmaf(a.w, c.z, acc[3][2]); acc[3][3] = fmaf(a.w, c.w, acc[3][3]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty * 4 + i, k = k0 + tx * 4 + j;
      if (m < M && k < K) atomicAdd(&dW[(size_t)m * K + k], acc[i][j]);
    }
}

// ================================================================================================================
// host side
// ================================================================================================================
inline dim3 grid_cb(int C, int B) { return dim3(C < 1024 ? C : 1024, B); }

#define LAUNCH_CHECK()      \
  do {                      \
    CTN_COUNT_LAUNCH();     \
    CTN_RETURN_IF_CUDA_ERR(); \
  } while (0)

struct TrainWs {
  // ---- saved by the forward
  float *w, *mask, *what, *skip;
  double *stats0, *stats;  // stats: [2*RX][B][2]
  std::vector<float*> x, hpre, upre;
  // ---- scratch (forward and backward)
  FoldedConv head;
  float *wimg, *Wcat, *Wt;
  float *T1, *G1, *G2;      // (B, H, pitch)
  float *r;                 // (B, Bc+Sc, pitch)
  float *dcat, *dS, *dxtmp; // (B, Bc+Sc, pitch), (B, Sc, pitch), (B, Bc, pitch)
  float *dwhat;             // (B, S*N, pitch)
  float *nA, *nB, *nC;      // (B, N, pitch): wn, d_wn, d_wprod
  float *sp, *dsp;          // (B, Sc, pitch)
  double* sums;             // (B, 2)
  size_t stats_bytes;
  void* tcn_mem;            // fp16-piece mode: state of the fused TCN forward (ctn_tcn_train_fwd)
  size_t tcn_bytes;
};

size_t max_wimg_bytes(const ctn_config_t* c) {
  if (c->math == CTN_MATH_FP32) return 256;
  const int N = c->n_basis, Bc = c->bottleneck, H = c->hidden, Sc = c->skip, SN = c->n_sources * c->n_basis;
  const int shapes[][2] = {{H, Bc}, {Bc + Sc, H}, {H, Bc + Sc}, {Bc, H}, {Bc, N}, {N, Bc}, {SN, Sc}, {Sc, SN}};
  size_t mx = 0;
  for (auto& s : shapes) {
    const size_t b = ctn_umma_wimg_bytes(s[0], s[1], c->math);
    if (b > mx) mx = b;
  }
  return mx;
}

void carve_train(Carver& cv, const ctn_config_t* c, int B, int pitch, TrainWs* ws) {
  const int RX = c->num_blocks * c->num_layers;
  const int N = c->n_basis, Bc = c->bottleneck, H = c->hidden, Sc = c->skip, S = c->n_sources;
  const size_t bp = (size_t)B * pitch;
  ws->stats0 = cv.take<double>((size_t)B * 2);
  ws->stats_bytes = sizeof(double) * 2 * RX * B * 2;
  ws->stats = cv.take<double>((size_t)2 * RX * B * 2);
  ws->sums = cv.take<double>((size_t)B * 2);
  ws->w = cv.take<float>(bp * N);
  ws->mask = cv.take<float>(bp * N * S);
  ws->what = cv.take<float>(bp * N * S);
  ws->skip = cv.take<float>(bp * Sc);
  ws->x.assign(RX, nullptr);
  ws->hpre.assign(RX, nullptr);
  ws->upre.assign(RX, nullptr);
  for (int i = 0; i < RX; ++i) {
    ws->x[i] = cv.take<float>(bp * Bc);
    ws->hpre[i] = cv.take<float>(bp * H);
    ws->upre[i] = cv.take<float>(bp * H);
  }
  ws->head.Wf = cv.take<float>((size_t)Bc * N);
  ws->head.v1 = cv.take<float>(Bc);
  ws->head.v2 = cv.take<float>(Bc);
  ws->head.vb = cv.take<float>(Bc);
  ws->tcn_mem = nullptr;
  ws->tcn_bytes = 0;
  if (c->math == CTN_MATH_F16X3 && c->sep_kernel == 3) {
    ws->tcn_bytes = ctn_tcn_train_ws_bytes(c, B, pitch);
    ws->tcn_mem = cv.take<char>(ws->tcn_bytes);
  }
  ws->wimg = cv.take<float>(max_wimg_bytes(c) / sizeof(float));
  size_t wmax = (size_t)(Bc + Sc) * H;
  if ((size_t)S * N * Sc > wmax) wmax = (size_t)S * N * Sc;
  if ((size_t)Bc * N > wmax) wmax = (size_t)Bc * N;
  ws->Wcat = cv.take<float>(wmax);
  ws->Wt = cv.take<float>(wmax);
  ws->T1 = cv.take<float>(bp * H);
  ws->G1 = cv.take<float>(bp * H);
  ws->G2 = cv.take<float>(bp * H);
  ws->r = cv.take<float>(bp * (Bc + Sc));
  ws->dcat = cv.take<float>(bp * (Bc + Sc));
  ws->dS = cv.take<float>(bp * Sc);
  ws->dxtmp = cv.take<float>(bp * Bc);
  ws->dwhat = cv.take<float>(bp * N * S);
  ws->nA = cv.take<float>(bp * N);
  ws->nB = cv.take<float>(bp * N);
  ws->nC = cv.take<float>(bp * N);
  ws->sp = cv.take<float>(bp * Sc);
  ws->dsp = cv.take<float>(bp * Sc);
}

int check_train_cfg(const ctn_config_t* c) {
  if (!c) return CTN_EINVAL;
  if (c->n_basis <= 0 || c->kernel_size <= 0 || c->stride <= 0 || c->n_sources <= 0 || c->bottleneck <= 0 || c->hidden <= 0 ||
      c->skip <= 0 || c->sep_kernel <= 0 || c->num_blocks <= 0 || c->num_layers <= 0)
    return CTN_EINVAL;
  if (c->kernel_size % c->stride != 0) return CTN_EINVAL;
  if (c->num_layers > 20 || c->num_blocks * c->num_layers > CTN_MAX_BLOCKS) return CTN_EUNSUPPORTED;
  if (c->causal || c->mask_softmax || c->in_channels > 1 || c->sep_kernel > CTN_MAX_P) return CTN_EUNSUPPORTED;  // softmax masks, multichannel: forward only
  if (c->math != CTN_MATH_FP32 && c->math != CTN_MATH_TF32X3 && c->math != CTN_MATH_TF32 && c->math != CTN_MATH_F16X3) return CTN_EINVAL;
  return CTN_OK;
}

// D (B, M, pitch) = W (M, K) . A (B, K, pitch), raw epilogue, in the configured numeric mode
// grad = true: the operand is a GRADIENT tensor.  Gradients have no fixed scale (1e-3 .. 1e-9 and below), which the fp16
// pieces of 'f16x3' cannot represent (subnormal below 6e-5, zero below 6e-8), so data-gradient contractions always use the
// tf32 pieces (8-bit exponent); 'f16x3' applies to the forward contractions, whose operands sit behind normalisations.
int gemm_raw(const ctn_config_t* c, TrainWs& ws, const float* W, int M, int K, const float* A, float* D, int B, int frames,
             int pitch, cudaStream_t st, bool grad = false) {
  PwArgs a;
  memset(&a, 0, sizeof(a));
  a.A = A; a.W = W; a.D = D; a.B = B; a.M = M; a.K = K; a.frames = frames; a.pitch = pitch;
  if (c->math == CTN_MATH_FP32) return ctn_pw_simt(a, PRO_NONE, EPI_RAW, st);
  // the training path keeps every contraction on the tf32 pieces: its forward operands (x_i, gLN2 output, skip sum) are
  // materialised tensors without the per-forward operand scales of the fused inference kernels (ctn_act_scales)
  (void)grad;
  const int math = c->math == CTN_MATH_F16X3 ? CTN_MATH_TF32X3 : c->math;
  CTN_TRY(ctn_umma_build_wimg(W, M, K, math, ws.wimg, st));
  a.wimg = ws.wimg;
  return ctn_pw_umma(a, PRO_NONE, EPI_RAW, math, st);
}

int transpose(const float* W, float* Wt, int M, int K, cudaStream_t st) {
  k_transpose<<<(M * K + 255) / 256, 256, 0, st>>>(W, Wt, M, K);
  LAUNCH_CHECK();
  return CTN_OK;
}

// dW (M, K) += sum dY X^T; rows [0, split_row) -> dWa, the rest -> dWb (nullable).  Tensor cores (3xTF32 / TF32) unless the
// configured mode is plain fp32, where the FFMA split-K kernel runs.
int wgrad(const ctn_config_t* c, const float* dy, size_t dy_bs, const float* x, size_t x_bs, float* dWa, float* dWb, int split_row,
          int M, int K, int B, int frames, int pitch, cudaStream_t st) {
  if (c->math != CTN_MATH_FP32)
    return ctn_wgrad_umma(dy, dy_bs, x, x_bs, dWa, dWb, split_row, M, K, B, frames, pitch, c->math, st);
  const int parts = dWb ? 2 : 1;
  for (int part = 0; part < parts; ++part) {
    const int r0 = part == 0 ? 0 : split_row, Mp = part == 0 ? (dWb ? split_row : M) : M - split_row;
    float* dW = part == 0 ? dWa : dWb;
    const float* dyp = dy + (size_t)r0 * pitch;
    const int tiles = ((Mp + 63) / 64) * ((K + 63) / 64);
    const long long total = (long long)B * ((frames + WG_T - 1) / WG_T);
    long long splits = (4 * 148 + tiles - 1) / tiles;
    if (splits > total) splits = total;
    if (splits < 1) splits = 1;
    const int upc = (int)((total + splits - 1) / splits);
    splits = (total + upc - 1) / upc;
    k_wgrad<<<dim3(tiles, (unsigned)splits), 256, 0, st>>>(dyp, dy_bs, x, x_bs, dW, Mp, K, B, frames, pitch, upc);
    LAUNCH_CHECK();
  }
  return CTN_OK;
}

int encdec_wgrad(const float* act, const float* sig, float* dW, int R, int N, int frames, int pitch, int T, int L, int stride,
                 int pad_left, cudaStream_t st) {
  if (L <= ENCDEC_MAX_L) {
    int gy = (4 * 148 + N - 1) / N;
    if (gy > R) gy = R;
    if (gy < 1) gy = 1;
    k_encdec_wgrad<<<dim3(N, gy), 256, 0, st>>>(act, sig, dW, R, N, frames, pitch, T, L, stride, pad_left);
  } else {
    k_encdec_wgrad_generic<<<dim3(L, N), 256, 0, st>>>(act, sig, dW, R, N, frames, pitch, T, L, stride, pad_left);
  }
  LAUNCH_CHECK();
  return CTN_OK;
}

int rowsum(const float* dy, size_t bs, int C, int B, int frames, int pitch, float* out, cudaStream_t st) {
  k_rowsum<<<dim3(C, B), 256, 0, st>>>(dy, bs, frames, pitch, out);
  LAUNCH_CHECK();
  return CTN_OK;
}

// gLN (+ optional PReLU in front) backward: dy (B,C,pitch) -> dpre (may alias dy); accumulates dgamma, dbeta, dslope, dbias
int gln_prelu_bwd(const float* dy, const float* pre, float* dpre, const float* slope, const float* g, const double* stats,
                  double n, float eps, double* sums, float* dgamma, float* dbeta, float* dslope, float* dbias, int B, int C,
                  int frames, int pitch, cudaStream_t st, bool reduced = false) {
  if (!reduced) {  // phase 1 (skipped when the producer of dy already accumulated sums / dgamma / dbeta)
    cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * 2 * B, st);
    if (e != cudaSuccess) return (int)e;
    k_gln_bwd_reduce<<<dim3(C, B), 256, 0, st>>>(dy, pre, slope, g, stats, n, eps, sums, dgamma, dbeta, C, frames, pitch);
    LAUNCH_CHECK();
  }
  k_gln_prelu_bwd_apply<<<dim3(C, B), 256, 0, st>>>(dy, pre, dpre, slope, g, stats, n, eps, sums, dslope, dbias, C, frames, pitch);
  LAUNCH_CHECK();
  return CTN_OK;
}

}  // namespace

extern "C" int ctn_train_workspace_bytes(const ctn_config_t* cfg, int batch, int T, size_t* bytes) {
  CTN_TRY(check_train_cfg(cfg));
  if (batch <= 0 || !bytes) return CTN_EINVAL;
  const int frames = ctn_frames(T, cfg->kernel_size, cfg->stride, nullptr, nullptr);
  if (frames <= 0) return CTN_EINVAL;
  Carver cv(nullptr);
  TrainWs ws;
  carve_train(cv, cfg, batch, ctn_pitch(frames), &ws);
  *bytes = cv.off + 256;
  return CTN_OK;
}

extern "C" int ctn_convtasnet_fwd_train(const ctn_config_t* c, const ctn_params_t* p, const float* x, int B, int T, float* out,
                                        void* train_ws, size_t train_ws_bytes, ctn_stream_t stream) {
  LaunchScope scope(x);
  CTN_TRY(check_train_cfg(c));
  if (!p || !p->blocks || !x || !out || !train_ws || B <= 0 || T <= 0) return CTN_EINVAL;
  if (((uintptr_t)train_ws) & 255) return CTN_EALIGN;
  size_t need = 0;
  CTN_TRY(ctn_train_workspace_bytes(c, B, T, &need));
  if (train_ws_bytes < need) return CTN_EWORKSPACE;
  int pl = 0, pr = 0;
  const int frames = ctn_frames(T, c->kernel_size, c->stride, &pl, &pr);
  const int pitch = ctn_pitch(frames);
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(train_ws);
  TrainWs ws;
  carve_train(cv, c, B, pitch, &ws);
  const int N = c->n_basis, Bc = c->bottleneck, H = c->hidden, Sc = c->skip, S = c->n_sources, R = c->num_blocks, X = c->num_layers;
  cudaError_t e = cudaMemsetAsync(ws.stats0, 0, sizeof(double) * 2 * B, st);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(ws.stats, 0, ws.stats_bytes, st);
  if (e != cudaSuccess) return (int)e;
  // encoder + gLN0 statistics (filterbank.py:222-229)
  CTN_TRY(ctn_encoder_fwd(x, p->enc_w, ws.w, B, T, pl, pr, N, c->kernel_size, c->stride, c->enc_relu, pitch, ws.stats0, stream));
  // head: x_0 = Wb gLN0(w) + bb (conv_tasnet.py:370-371), gLN0 folded into the contraction like the inference path
  {
    CTN_TRY(ctn_fold_conv(p->bn_w, p->bn_b, p->norm0_g, p->norm0_b, Bc, N, ws.head, 0, st, sqrtf((float)N * (float)frames) * 1.0001f));
    PwArgs a;
    memset(&a, 0, sizeof(a));
    a.A = ws.w; a.W = ws.head.Wf; a.D = ws.x[0]; a.B = B; a.M = Bc; a.K = N; a.frames = frames; a.pitch = pitch;
    a.v1 = ws.head.v1; a.v2 = ws.head.v2; a.stats_in = ws.stats0; a.n_in = (double)N * (double)frames; a.eps = c->eps;
    if (c->math == CTN_MATH_FP32) {
      CTN_TRY(ctn_pw_simt(a, PRO_NONE, EPI_HEAD, st));
    } else {
      // the head reads the un-normalised encoder output: tf32 pieces even in the fp16-piece mode (see ctn_api.cu)
      const int head_math = c->math == CTN_MATH_F16X3 ? CTN_MATH_TF32X3 : c->math;
      CTN_TRY(ctn_umma_build_wimg(ws.head.Wf, Bc, N, head_math, ws.wimg, st));
      a.wimg = ws.wimg;
      CTN_TRY(ctn_pw_umma(a, PRO_NONE, EPI_HEAD, head_math, st));
    }
  }
  const double nH = (double)H * (double)frames;
  // un-normalised operands (x_i, skip sum) without operand scales: tf32 pieces (8-bit exponent) in the fp16-piece mode
  const int fmath = c->math == CTN_MATH_F16X3 ? CTN_MATH_TF32X3 : c->math;
  // fp16-piece mode: the TCN runs through the SAME fused TMA-fed kernels as inference (pw1 with the residual update fused,
  // depthwise producer feeding the [out;skip] contraction), which additionally leave x_i, W1 x + b1 and the depthwise
  // pre-activation behind for the backward -- 2 launches per block instead of 7, no u / gLN2(u) round trips
  bool fused = false;
  const float* mask_scale = nullptr;
  if (ws.tcn_mem) {
    TcnTrainHooks hk{ws.x.data(), ws.hpre.data(), ws.upre.data()};
    const int rc = ctn_tcn_train_fwd(c, p->blocks, ws.tcn_mem, ws.tcn_bytes, &hk, ws.stats, ws.skip, ws.head.vb, Bc, p->prelu_out, &mask_scale,
                                     B, frames, pitch, st);
    if (rc == CTN_OK) fused = true;
    else if (rc != CTN_EUNSUPPORTED) return rc;
    else if ((e = cudaMemsetAsync(ws.stats, 0, ws.stats_bytes, st)) != cudaSuccess) return (int)e;  // shapes outside the fused envelope
  }
  for (int i = 0; i < (fused ? 0 : R * X); ++i) {
    const ctn_block_params_t& q = p->blocks[i];
    const bool has_out = q.out_w != nullptr;
    if (!has_out && i != R * X - 1) return CTN_EINVAL;
    const int dil = 1 << (i % X);
    const int pad_left = ((c->sep_kernel - 1) * dil) / 2;
    double* st1 = ws.stats + (size_t)(2 * i) * B * 2;
    double* st2 = ws.stats + (size_t)(2 * i + 1) * B * 2;
    // h_pre = W1 x + b1 ; stats1 of PReLU(h_pre)
    if (c->math == CTN_MATH_FP32) {
      CTN_TRY(gemm_raw(c, ws, q.bottleneck_w, H, Bc, ws.x[i], ws.hpre[i], B, frames, pitch, st));
      k_bias_prelu_stats<<<grid_cb(H, B), 256, 0, st>>>(ws.hpre[i], q.bottleneck_b, q.prelu1, st1, H, frames, pitch);
      LAUNCH_CHECK();
    } else {  // bias, PReLU statistics fused into the contraction's epilogue; the PRE-activation is what gets stored
      PwArgs a;
      memset(&a, 0, sizeof(a));
      a.A = ws.x[i]; a.W = q.bottleneck_w; a.D = ws.hpre[i]; a.B = B; a.M = H; a.K = Bc; a.frames = frames; a.pitch = pitch;
      a.bias = q.bottleneck_b; a.slope = q.prelu1; a.stats_out = st1; a.store_pre = 1;
      CTN_TRY(ctn_umma_build_wimg(q.bottleneck_w, H, Bc, fmath, ws.wimg, st));
      a.wimg = ws.wimg;
      CTN_TRY(ctn_pw_umma(a, PRO_NONE, EPI_H, fmath, st));
    }
    // u_pre = dwconv(gLN1(PReLU(h_pre))) + bd ; stats2 of PReLU(u_pre)
    k_dw_train_fwd<<<grid_cb(H, B), 256, 0, st>>>(ws.hpre[i], ws.upre[i], q.norm1_g, q.norm1_b, q.dw_w, q.dw_b, q.prelu1, q.prelu2,
                                                  st1, st2, H, frames, pitch, c->sep_kernel, dil, pad_left, nH, c->eps_tcn);
    LAUNCH_CHECK();
    // un = gLN2(PReLU(u_pre)) ; r = [Wo; Ws] un
    k_act_norm<<<grid_cb(H, B), 256, 0, st>>>(ws.upre[i], ws.T1, q.prelu2, q.norm2_g, q.norm2_b, st2, nH, c->eps_tcn, H, frames, pitch);
    LAUNCH_CHECK();
    const int Mt = has_out ? Bc + Sc : Sc;
    if (has_out) {
      if ((e = cudaMemcpyAsync(ws.Wcat, q.out_w, sizeof(float) * (size_t)Bc * H, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return (int)e;
    }
    if ((e = cudaMemcpyAsync(ws.Wcat + (has_out ? (size_t)Bc * H : 0), q.skip_w, sizeof(float) * (size_t)Sc * H, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return (int)e;
    CTN_TRY(gemm_raw(c, ws, ws.Wcat, Mt, H, ws.T1, ws.r, B, frames, pitch, st));
    // x_{i+1} = x_i + out + bo ; skip += skip_i + bs
    k_res_skip<<<grid_cb(Mt, B), 256, 0, st>>>(ws.r, Mt, ws.x[i], has_out ? ws.x[i + 1] : nullptr, ws.skip, q.out_b, q.skip_b, Bc, Sc,
                                               has_out ? 1 : 0, i == 0 ? 1 : 0, frames, pitch);
    LAUNCH_CHECK();
  }
  // tail: PReLU -> mask 1x1 -> sigmoid -> * w (conv_tasnet.py:373-376, 158-160); keeps the mask
  {
    PwArgs a;
    memset(&a, 0, sizeof(a));
    a.A = ws.skip; a.W = p->mask_w; a.D = ws.what; a.B = B; a.M = S * N; a.K = Sc; a.frames = frames; a.pitch = pitch;
    a.pro_slope = p->prelu_out; a.bias = p->mask_b; a.wenc = ws.w; a.Nb = N; a.mask_out = ws.mask;
    if (c->math == CTN_MATH_FP32) {
      CTN_TRY(ctn_pw_simt(a, PRO_PRELU, EPI_MASK, st));
    } else {
      const int mmath = fused ? CTN_MATH_F16X3 : fmath;  // the fused forward also produced the operand scale of PReLU(skip sum)
      if (fused) a.act_scale = mask_scale;
      CTN_TRY(ctn_umma_build_wimg(p->mask_w, S * N, Sc, mmath, ws.wimg, st));
      a.wimg = ws.wimg;
      CTN_TRY(ctn_pw_umma(a, PRO_PRELU, EPI_MASK, mmath, st));
    }
  }
  CTN_TRY(ctn_decoder_fwd(ws.what, p->dec_w, out, B * S, N, frames, pitch, c->kernel_size, c->stride, pl, T, stream));
  return CTN_OK;
}

// grads: same layout as params; every tensor must be ZERO on entry (the kernels accumulate with atomics)
extern "C" int ctn_convtasnet_bwd(const ctn_config_t* c, const ctn_params_t* p, const ctn_params_t* grads, const float* x,
                                  const float* d_out, int B, int T, void* train_ws, size_t train_ws_bytes, ctn_stream_t stream) {
  LaunchScope scope(x);
  CTN_TRY(check_train_cfg(c));
  if (!p || !p->blocks || !grads || !grads->blocks || !x || !d_out || !train_ws || B <= 0 || T <= 0) return CTN_EINVAL;
  if (((uintptr_t)train_ws) & 255) return CTN_EALIGN;
  size_t need = 0;
  CTN_TRY(ctn_train_workspace_bytes(c, B, T, &need));
  if (train_ws_bytes < need) return CTN_EWORKSPACE;
  int pl = 0, pr = 0;
  const int frames = ctn_frames(T, c->kernel_size, c->stride, &pl, &pr);
  const int pitch = ctn_pitch(frames);
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(train_ws);
  TrainWs ws;
  carve_train(cv, c, B, pitch, &ws);
  const int N = c->n_basis, Bc = c->bottleneck, H = c->hidden, Sc = c->skip, S = c->n_sources, RX = c->num_blocks * c->num_layers,
            X = c->num_layers, L = c->kernel_size;
  const size_t bsN = (size_t)N * pitch, bsH = (size_t)H * pitch, bsBc = (size_t)Bc * pitch, bsSc = (size_t)Sc * pitch,
               bsCat = (size_t)(Bc + Sc) * pitch, bsSN = (size_t)S * N * pitch;
  const double nH = (double)H * (double)frames;
  auto G = [](const float* q) { return const_cast<float*>(q); };

  // ---- decoder (filterbank.py:243-249): d_what = conv1d(d_out; Wd) (the transposed conv's adjoint), dWd
  CTN_TRY(ctn_encoder_fwd(d_out, p->dec_w, ws.dwhat, B * S, T, pl, pr, N, L, c->stride, 0, pitch, nullptr, stream));
  CTN_TRY(encdec_wgrad(ws.what, d_out, G(grads->dec_w), B * S, N, frames, pitch, T, L, c->stride, pl, st));
  // ---- w_hat = w * sigmoid(m_pre): d_mpre (in place), d_wprod
  k_mask_bwd<<<grid_cb(N, B), 256, 0, st>>>(ws.dwhat, ws.w, ws.mask, ws.nC, S, N, frames, pitch);
  LAUNCH_CHECK();
  // ---- mask conv (conv_tasnet.py:341,374): dWm, dbm, d_sp = Wm^T d_mpre
  k_prelu_apply<<<grid_cb(Sc, B), 256, 0, st>>>(ws.skip, ws.sp, p->prelu_out, Sc, frames, pitch);
  LAUNCH_CHECK();
  CTN_TRY(wgrad(c, ws.dwhat, bsSN, ws.sp, bsSc, G(grads->mask_w), nullptr, 0, S * N, Sc, B, frames, pitch, st));
  CTN_TRY(rowsum(ws.dwhat, bsSN, S * N, B, frames, pitch, G(grads->mask_b), st));
  CTN_TRY(transpose(p->mask_w, ws.Wt, S * N, Sc, st));
  CTN_TRY(gemm_raw(c, ws, ws.Wt, Sc, S * N, ws.dwhat, ws.dsp, B, frames, pitch, st, /*grad=*/true));
  // ---- PReLU on the skip sum (conv_tasnet.py:340,373): dS (the gradient of EVERY block's skip output)
  k_prelu_bwd<<<dim3(Sc, B), 256, 0, st>>>(ws.dsp, ws.skip, ws.dS, p->prelu_out, G(grads->prelu_out), Sc, frames, pitch);
  LAUNCH_CHECK();
  // dcat rows [Bc, Bc+Sc) = dS for all blocks with an output head; rows [0,Bc) = gradient of the block's residual output
  k_rows<<<grid_cb(Sc, B), 256, 0, st>>>(ws.dcat + bsBc, bsCat, ws.dS, bsSc, Sc, 0, frames, pitch);
  LAUNCH_CHECK();
  // ---- residual blocks, last to first
  for (int i = RX - 1; i >= 0; --i) {
    const ctn_block_params_t& q = p->blocks[i];
    const ctn_block_params_t& gq = grads->blocks[i];
    const bool has_out = q.out_w != nullptr;
    const int dil = 1 << (i % X);
    const int pad_left = ((c->sep_kernel - 1) * dil) / 2;
    const double* st1 = ws.stats + (size_t)(2 * i) * B * 2;
    const double* st2 = ws.stats + (size_t)(2 * i + 1) * B * 2;
    const int Mt = has_out ? Bc + Sc : Sc;
    const float* dY = has_out ? ws.dcat : ws.dS;  // (B, Mt, pitch)
    const size_t dY_bs = has_out ? bsCat : bsSc;
    // un = gLN2(PReLU(u_pre)) recomputed for the weight gradients of the two heads
    k_act_norm<<<grid_cb(H, B), 256, 0, st>>>(ws.upre[i], ws.T1, q.prelu2, q.norm2_g, q.norm2_b, st2, nH, c->eps_tcn, H, frames, pitch);
    LAUNCH_CHECK();
    if (has_out) {
      CTN_TRY(wgrad(c, dY, dY_bs, ws.T1, bsH, G(gq.out_w), G(gq.skip_w), Bc, Bc + Sc, H, B, frames, pitch, st));
      CTN_TRY(rowsum(dY, dY_bs, Bc, B, frames, pitch, G(gq.out_b), st));
    } else {
      CTN_TRY(wgrad(c, dY, dY_bs, ws.T1, bsH, G(gq.skip_w), nullptr, 0, Sc, H, B, frames, pitch, st));
    }
    const float* dYs = dY + (has_out ? bsBc : 0);
    CTN_TRY(rowsum(dYs, dY_bs, Sc, B, frames, pitch, G(gq.skip_b), st));
    // d_un = [Wo; Ws]^T dY
    {
      cudaError_t e;
      if (has_out && (e = cudaMemcpyAsync(ws.Wcat, q.out_w, sizeof(float) * (size_t)Bc * H, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return (int)e;
      if ((e = cudaMemcpyAsync(ws.Wcat + (has_out ? (size_t)Bc * H : 0), q.skip_w, sizeof(float) * (size_t)Sc * H, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return (int)e;
    }
    CTN_TRY(transpose(ws.Wcat, ws.Wt, Mt, H, st));
    CTN_TRY(gemm_raw(c, ws, ws.Wt, H, Mt, dY, ws.G1, B, frames, pitch, st, /*grad=*/true));
    // gLN2 + PReLU2 backward -> d_u_pre (G1 in place); dgamma2, dbeta2, da2, d(bd)
    CTN_TRY(gln_prelu_bwd(ws.G1, ws.upre[i], ws.G1, q.prelu2, q.norm2_g, st2, nH, c->eps_tcn, ws.sums, G(gq.norm2_g), G(gq.norm2_b),
                          G(gq.prelu2), G(gq.dw_b), B, H, frames, pitch, st));
    // depthwise conv backward -> d_hn (G2), d(wd); fused: phase 1 of the gLN1 backward (per-sample sums, dgamma1, dbeta1)
    {
      cudaError_t e = cudaMemsetAsync(ws.sums, 0, sizeof(double) * 2 * B, st);
      if (e != cudaSuccess) return (int)e;
    }
    k_dw_bwd<<<dim3(H, B), 256, 0, st>>>(ws.G1, ws.hpre[i], ws.G2, q.prelu1, q.norm1_g, q.norm1_b, st1, nH, c->eps_tcn, q.dw_w,
                                         G(gq.dw_w), ws.sums, G(gq.norm1_g), G(gq.norm1_b), H, frames, pitch, c->sep_kernel, dil,
                                         pad_left);
    LAUNCH_CHECK();
    // gLN1 + PReLU1 backward, phase 2 -> d_h_pre (G2 in place); da1, db1
    CTN_TRY(gln_prelu_bwd(ws.G2, ws.hpre[i], ws.G2, q.prelu1, q.norm1_g, st1, nH, c->eps_tcn, ws.sums, G(gq.norm1_g), G(gq.norm1_b),
                          G(gq.prelu1), G(gq.bottleneck_b), B, H, frames, pitch, st, /*reduced=*/true));
    // bottleneck 1x1: dW1 = d_h_pre x_i^T ; d_x_i = W1^T d_h_pre (+ residual path)
    CTN_TRY(wgrad(c, ws.G2, bsH, ws.x[i], bsBc, G(gq.bottleneck_w), nullptr, 0, H, Bc, B, frames, pitch, st));
    CTN_TRY(transpose(q.bottleneck_w, ws.Wt, H, Bc, st));
    CTN_TRY(gemm_raw(c, ws, ws.Wt, Bc, H, ws.G2, ws.dxtmp, B, frames, pitch, st, /*grad=*/true));
    k_rows<<<grid_cb(Bc, B), 256, 0, st>>>(ws.dcat, bsCat, ws.dxtmp, bsBc, Bc, has_out ? 1 : 0, frames, pitch);
    LAUNCH_CHECK();
  }
  // ---- head (conv_tasnet.py:333-335,370-371): x_0 = Wb gLN0(w) + bb.   d_x0 = dcat rows [0,Bc)
  k_act_norm<<<grid_cb(N, B), 256, 0, st>>>(ws.w, ws.nA, nullptr, p->norm0_g, p->norm0_b, ws.stats0, (double)N * frames, c->eps, N,
                                            frames, pitch);
  LAUNCH_CHECK();
  CTN_TRY(wgrad(c, ws.dcat, bsCat, ws.nA, bsN, G(grads->bn_w), nullptr, 0, Bc, N, B, frames, pitch, st));
  CTN_TRY(rowsum(ws.dcat, bsCat, Bc, B, frames, pitch, G(grads->bn_b), st));
  // d_wn = Wb^T d_x0 (the operand of the contraction must be dense (B, K, pitch): copy the rows out of dcat)
  k_rows<<<grid_cb(Bc, B), 256, 0, st>>>(ws.dxtmp, bsBc, ws.dcat, bsCat, Bc, 0, frames, pitch);
  LAUNCH_CHECK();
  CTN_TRY(transpose(p->bn_w, ws.Wt, Bc, N, st));
  CTN_TRY(gemm_raw(c, ws, ws.Wt, N, Bc, ws.dxtmp, ws.nB, B, frames, pitch, st, /*grad=*/true));
  // gLN0 backward -> d_w (norm path) ; + product path ; ReLU mask of the encoder if any
  CTN_TRY(gln_prelu_bwd(ws.nB, ws.w, ws.nB, nullptr, p->norm0_g, ws.stats0, (double)N * frames, c->eps, ws.sums, G(grads->norm0_g),
                        G(grads->norm0_b), nullptr, nullptr, B, N, frames, pitch, st));
  k_dw_combine<<<grid_cb(N, B), 256, 0, st>>>(ws.nB, ws.nC, ws.w, c->enc_relu, N, frames, pitch);
  LAUNCH_CHECK();
  // ---- encoder (filterbank.py:212,222): dWe
  CTN_TRY(encdec_wgrad(ws.nB, x, G(grads->enc_w), B, N, frames, pitch, T, L, c->stride, pl, st));
  return CTN_OK;
}
