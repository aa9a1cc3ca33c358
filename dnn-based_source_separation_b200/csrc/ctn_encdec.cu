// Encoder (strided 1-D conv) and decoder (transposed conv, overlap-add) kernels.  HBM-bound:
//   encoder writes N*frames floats per sample (262 MB at cfg2), decoder reads S*N*frames floats.
// Lanes run along time so every global access is a 128-byte coalesced row segment; the 16-tap filter bank
// lives transposed in shared memory and is read with broadcast 128-bit LDS.
#include <stdlib.h>
#include "ctn_common.cuh"

// ------------------------------------------------------------------------------------------------
// Encoder: w[b][n][f] = sum_k W[n][k] * xpad[b][f*stride + k]      (src/models/filterbank.py:222-229)
// grid (pitch/128, B), block 128: thread = frame; loops over n in groups of 4.
// ------------------------------------------------------------------------------------------------
template <int L>
__global__ void __launch_bounds__(128) k_encoder(const float* __restrict__ x, const float* __restrict__ W,
                                                 float* __restrict__ w, int T, int pad_left, int N, int stride,
                                                 int frames, int pitch, int relu, double* __restrict__ stats) {
  extern __shared__ float sm[];
  float* Wt = sm;                       // [L][N4]  (N4 = N rounded up to 4)
  const int N4 = (N + 3) & ~3;
  float* xs = sm + L * N4;              // [127*stride + L]
  __shared__ double red[64];
  const int b = blockIdx.y, f0 = blockIdx.x * 128, tid = threadIdx.x;
  for (int i = tid; i < L * N4; i += 128) {
    const int k = i / N4, n = i - k * N4;
    Wt[i] = n < N ? W[n * L + k] : 0.f;
  }
  const int seg = 127 * stride + L;
  const float* xb = x + (size_t)b * T;
  for (int i = tid; i < seg; i += 128) {
    const int t = f0 * stride + i - pad_left;
    xs[i] = (t >= 0 && t < T) ? xb[t] : 0.f;
  }
  __syncthreads();
  float xw[L];
#pragma unroll
  for (int k = 0; k < L; ++k) xw[k] = xs[tid * stride + k];
  const int f = f0 + tid;
  const bool valid = f < frames;
  const bool inb = f < pitch;
  float* wb = w + (size_t)b * N * pitch + (inb ? f : 0);
  double s = 0.0, ss = 0.0;
  float ls = 0.f, lss = 0.f;
  for (int n = 0; n < N; n += 4) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int k = 0; k < L; ++k) {
      const float4 wv = *reinterpret_cast<const float4*>(&Wt[k * N4 + n]);
      a0 = fmaf(wv.x, xw[k], a0);
      a1 = fmaf(wv.y, xw[k], a1);
      a2 = fmaf(wv.z, xw[k], a2);
      a3 = fmaf(wv.w, xw[k], a3);
    }
    if (relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); a2 = fmaxf(a2, 0.f); a3 = fmaxf(a3, 0.f); }
    if (!valid) { a0 = a1 = a2 = a3 = 0.f; }
    if (inb) wb[(size_t)n * pitch] = a0;
    if (n + 1 < N) { if (inb) wb[(size_t)(n + 1) * pitch] = a1; } else a1 = 0.f;
    if (n + 2 < N) { if (inb) wb[(size_t)(n + 2) * pitch] = a2; } else a2 = 0.f;
    if (n + 3 < N) { if (inb) wb[(size_t)(n + 3) * pitch] = a3; } else a3 = 0.f;
    ls += (a0 + a1) + (a2 + a3);
    lss += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    if ((n & 63) == 60) { s += ls; ss += lss; ls = 0.f; lss = 0.f; }  // spill fp32 partials to double
  }
  if (stats != nullptr) {
    s += ls; ss += lss;
    block_sum2_d(s, ss, red);
    if (tid == 0) { atomicAdd(&stats[2 * b], s); atomicAdd(&stats[2 * b + 1], ss); }
  }
}

// Fast path (kernel = 2 x stride: the Conv-TasNet / DPRNN-TasNet encoders): thread = 4 consecutive frames x 4 channels per step, so
// one broadcast LDS.128 of the filter bank feeds 16 FMAs (the kernel above issues one per 4) and every store is a 128-bit STG -- a
// warp writes 512 contiguous bytes of one channel row.  Block = 128 frames x all N channels, 4 warps each owning a quarter of the
// channels; gLN statistics per thread in fp32 (<= 64 values), then double.
template <int L, int STRIDE>
__global__ void __launch_bounds__(128) k_encoder_v4(const float* __restrict__ x, const float* __restrict__ W, float* __restrict__ w, int T,
                                                    int pad_left, int N, int frames, int pitch, int relu, double* __restrict__ stats) {
  constexpr int XW = 3 * STRIDE + L;  // input samples under 4 consecutive frames
  extern __shared__ float sm[];
  const int N4 = (N + 3) & ~3;
  float* Wt = sm;                     // [L][N4]
  float* xs = sm + L * N4;            // [127*STRIDE + L]
  __shared__ double red[64];
  const int b = blockIdx.y, f0 = blockIdx.x * 128, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < L * N4; i += 128) {
    const int k = i / N4, n = i - k * N4;
    Wt[i] = n < N ? W[n * L + k] : 0.f;
  }
  const int seg = 127 * STRIDE + L;
  const float* xb = x + (size_t)b * T;
  for (int i = tid; i < seg; i += 128) {
    const int t = f0 * STRIDE + i - pad_left;
    xs[i] = (t >= 0 && t < T) ? xb[t] : 0.f;
  }
  __syncthreads();
  float xw[XW];
#pragma unroll
  for (int k = 0; k < XW; ++k) xw[k] = xs[lane * 4 * STRIDE + k];
  const int f = f0 + lane * 4;
  const bool v0 = f < frames, v1 = f + 1 < frames, v2 = f + 2 < frames, v3 = f + 3 < frames;
  const int nq = ((N4 / 4 + 3) / 4) * 4;  // channels per warp, a multiple of 4
  const int n_beg = warp * nq, n_end = min(N, n_beg + nq);
  double s = 0.0, ss = 0.0;
  float ls = 0.f, lss = 0.f;
  int since = 0;
  for (int n = n_beg; n < n_end; n += 4) {
    float a[4][4];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int q = 0; q < 4; ++q) a[c][q] = 0.f;
#pragma unroll
    for (int k = 0; k < L; ++k) {
      const float4 wv = *reinterpret_cast<const float4*>(&Wt[k * N4 + n]);
      const float wc[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int q = 0; q < 4; ++q) a[c][q] = fmaf(wc[c], xw[q * STRIDE + k], a[c][q]);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (n + c >= N) break;
      float4 o = make_float4(a[c][0], a[c][1], a[c][2], a[c][3]);
      if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
      if (!v0) o.x = 0.f;
      if (!v1) o.y = 0.f;
      if (!v2) o.z = 0.f;
      if (!v3) o.w = 0.f;
      *reinterpret_cast<float4*>(w + ((size_t)b * N + n + c) * pitch + f) = o;
      ls += (o.x + o.y) + (o.z + o.w);
      lss = fmaf(o.x, o.x, fmaf(o.y, o.y, fmaf(o.z, o.z, fmaf(o.w, o.w, lss))));
    }
    if (++since == 4) { s += ls; ss += lss; ls = 0.f; lss = 0.f; since = 0; }  // spill fp32 partials (<= 64 values) to double
  }
  if (stats != nullptr) {
    s += ls; ss += lss;
    block_sum2_d(s, ss, red);
    if (tid == 0) { atomicAdd(&stats[2 * b], s); atomicAdd(&stats[2 * b + 1], ss); }
  }
}

template <int L>
static int launch_encoder(const float* x, const float* W, float* w, int B, int T, int pad_left, int N, int stride,
                          int frames, int pitch, int relu, double* stats, cudaStream_t st) {
  const int N4 = (N + 3) & ~3;
  const size_t smem = sizeof(float) * ((size_t)L * N4 + 127 * stride + L);
  if (smem > 200 * 1024) return CTN_EUNSUPPORTED;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_encoder<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  dim3 grid((pitch + 127) / 128, B);
  if constexpr (L <= 20) {  // longer kernels: the 3*stride + L input window no longer fits the register file
  if (stride * 2 == L && pitch % 128 == 0 && (((uintptr_t)w) & 15) == 0) {
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(k_encoder_v4<L, L / 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
    }
    k_encoder_v4<L, L / 2><<<grid, 128, smem, st>>>(x, W, w, T, pad_left, N, frames, pitch, relu, stats);
    CTN_COUNT_LAUNCH();
    CTN_RETURN_IF_CUDA_ERR();
    return CTN_OK;
  }
  }
  k_encoder<L><<<grid, 128, smem, st>>>(x, W, w, T, pad_left, N, stride, frames, pitch, relu, stats);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

extern "C" int ctn_encoder_fwd(const float* x, const float* enc_w, float* w, int B, int T, int pad_left, int pad_right,
                               int N, int L, int stride, int relu, int w_pitch, double* stats, ctn_stream_t stream) {
  LaunchScope scope(w);
  if (!x || !enc_w || !w || B <= 0 || T <= 0 || N <= 0 || L <= 0 || stride <= 0) return CTN_EINVAL;
  const int Tp = T + pad_left + pad_right;
  if (Tp < L || (Tp - L) % stride != 0) return CTN_EINVAL;
  const int frames = (Tp - L) / stride + 1;
  if (w_pitch < frames) return CTN_EALIGN;
  cudaStream_t st = (cudaStream_t)stream;
#define ENC_CASE(LL) case LL: return launch_encoder<LL>(x, enc_w, w, B, T, pad_left, N, stride, frames, w_pitch, relu, stats, st)
  switch (L) {
    ENC_CASE(2); ENC_CASE(4); ENC_CASE(8); ENC_CASE(16); ENC_CASE(20); ENC_CASE(32); ENC_CASE(40); ENC_CASE(64);
    default: return CTN_EUNSUPPORTED;
  }
#undef ENC_CASE
}

// ------------------------------------------------------------------------------------------------
// Decoder: full[bs][j*stride + q] = sum_{r<R} sum_n what[bs][n][j-r] * Wd[n][r*stride + q]
//          (ConvTranspose1d, src/models/filterbank.py:245-247), R = L/stride overlapping frames.
// thread = output segment j (stride consecutive samples); grid (ceil(nseg/128), BS), block 128.
// The crop of src/models/conv_tasnet.py:169 is fused: y[t] = full[t + crop_left].
// ------------------------------------------------------------------------------------------------
// The channel sum is split over DEC_SPLIT thread groups of a block (each walks N/DEC_SPLIT channels with its own
// accumulators, partial sums meet in shared memory): 4x the loads in flight per SM of a thread-per-segment kernel, which
// was latency-bound at ~1 TB/s (2048 resident threads instead of 896).
constexpr int DEC_SPLIT = 4;
template <int STRIDE, int R>
__global__ void __launch_bounds__(128 * DEC_SPLIT) k_decoder(const float* __restrict__ what, const float* __restrict__ Wd,
                                                             float* __restrict__ y, int N, int frames, int in_pitch,
                                                             int crop_left, int T_out) {
  constexpr int L = STRIDE * R;
  extern __shared__ float sm[];  // Wd as [N][L], then the partial sums [DEC_SPLIT-1][STRIDE][128]
  float* red = sm + (size_t)N * L;
  const int tid = threadIdx.x, bs = blockIdx.y;
  const int seg = tid & 127, part = tid >> 7;
  for (int i = tid; i < N * L; i += 128 * DEC_SPLIT) sm[i] = Wd[i];
  __syncthreads();
  const int j = blockIdx.x * 128 + seg;  // segment index, 0 .. frames+R-2
  const float* wb = what + (size_t)bs * N * in_pitch;
  float acc[STRIDE];
#pragma unroll
  for (int q = 0; q < STRIDE; ++q) acc[q] = 0.f;
  bool ok[R];
#pragma unroll
  for (int r = 0; r < R; ++r) ok[r] = (j - r) >= 0 && (j - r) < frames;
  const int nper = (N + DEC_SPLIT - 1) / DEC_SPLIT;
  const int n_begin = part * nper, n_end = min(N, n_begin + nper);
  for (int n = n_begin; n < n_end; ++n) {
    const float* wrow = wb + (size_t)n * in_pitch;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float v = ok[r] ? __ldg(wrow + (j - r)) : 0.f;
#pragma unroll
      for (int q = 0; q < STRIDE; ++q) acc[q] = fmaf(v, sm[n * L + r * STRIDE + q], acc[q]);
    }
  }
  if (part > 0) {
#pragma unroll
    for (int q = 0; q < STRIDE; ++q) red[((part - 1) * STRIDE + q) * 128 + seg] = acc[q];
  }
  __syncthreads();
  if (part == 0) {
    float* yb = y + (size_t)bs * T_out;
#pragma unroll
    for (int q = 0; q < STRIDE; ++q) {
      float v = acc[q];
#pragma unroll
      for (int p2 = 0; p2 < DEC_SPLIT - 1; ++p2) v += red[(p2 * STRIDE + q) * 128 + seg];
      const int t = j * STRIDE + q - crop_left;
      if (t >= 0 && t < T_out && j < frames + R - 1) yb[t] = v;
    }
  }
}

// generic fallback: thread = output sample
__global__ void __launch_bounds__(128) k_decoder_generic(const float* __restrict__ what, const float* __restrict__ Wd,
                                                         float* __restrict__ y, int N, int frames, int in_pitch, int L,
                                                         int stride, int crop_left, int T_out) {
  const int bs = blockIdx.y;
  const int t = blockIdx.x * 128 + threadIdx.x;
  if (t >= T_out) return;
  const int tf = t + crop_left;
  const int R = L / stride;
  const int j = tf / stride, q = tf - j * stride;
  const float* wb = what + (size_t)bs * N * in_pitch;
  float acc = 0.f;
  for (int r = 0; r < R; ++r) {
    const int f = j - r;
    if (f < 0 || f >= frames) continue;
    for (int n = 0; n < N; ++n) acc = fmaf(__ldg(wb + (size_t)n * in_pitch + f), __ldg(Wd + n * L + r * stride + q), acc);
  }
  y[(size_t)bs * T_out + t] = acc;
}

template <int STRIDE, int R>
static int launch_decoder(const float* what, const float* Wd, float* y, int BS, int N, int frames, int in_pitch,
                          int crop_left, int T_out, cudaStream_t st) {
  const size_t smem = sizeof(float) * ((size_t)N * STRIDE * R + (size_t)(DEC_SPLIT - 1) * STRIDE * 128);
  if (smem > 200 * 1024) return CTN_EUNSUPPORTED;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_decoder<STRIDE, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  const int nseg = frames + R - 1;
  dim3 grid((nseg + 127) / 128, BS);
  k_decoder<STRIDE, R><<<grid, 128 * DEC_SPLIT, smem, st>>>(what, Wd, y, N, frames, in_pitch, crop_left, T_out);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

extern "C" int ctn_decoder_fwd(const float* w_hat, const float* dec_w, float* y, int BS, int N, int frames,
                               int in_pitch, int L, int stride, int crop_left, int T_out, ctn_stream_t stream) {
  LaunchScope scope(w_hat);
  if (!w_hat || !dec_w || !y || BS <= 0 || N <= 0 || frames <= 0 || L <= 0 || stride <= 0 || L % stride != 0)
    return CTN_EINVAL;
  if (in_pitch < frames) return CTN_EINVAL;
  const int full = (frames - 1) * stride + L;
  if (crop_left < 0 || T_out <= 0 || crop_left + T_out > full) return CTN_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const int R = L / stride;
  if (stride == 8 && R == 2) return launch_decoder<8, 2>(w_hat, dec_w, y, BS, N, frames, in_pitch, crop_left, T_out, st);
  if (stride == 1 && R == 2) return launch_decoder<1, 2>(w_hat, dec_w, y, BS, N, frames, in_pitch, crop_left, T_out, st);
  if (stride == 10 && R == 2) return launch_decoder<10, 2>(w_hat, dec_w, y, BS, N, frames, in_pitch, crop_left, T_out, st);
  if (stride == 2 && R == 2) return launch_decoder<2, 2>(w_hat, dec_w, y, BS, N, frames, in_pitch, crop_left, T_out, st);
  dim3 grid((T_out + 127) / 128, BS);
  k_decoder_generic<<<grid, 128, 0, st>>>(w_hat, dec_w, y, N, frames, in_pitch, L, stride, crop_left, T_out);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

// ------------------------------------------------------------------------------------------------
// Multichannel filter banks (in_channels = n_mics > 1: the 4-D input form of conv_tasnet.py:138-141, 167-168; MUSDB18 recipes).
// Forward only, straightforward kernels (thread = frame / output sample): this is the widened input format, not the measured path.
//   encoder: w[b][n][f] = sum_c sum_k W[n][c][k] * xpad[b][c][f*stride + k]      (Conv1d(C, N, L, stride), filterbank.py:212,222-229)
//   decoder: y[bs][c][t] = sum_n sum_{f,k: f*stride + k = t + crop} what[bs][n][f] * Wd[n][c][k]  (ConvTranspose1d(N, C, L, stride))
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_encoder_mc(const float* __restrict__ x, const float* __restrict__ W, float* __restrict__ w, int C,
                                                    int T, int pad_left, int N, int L, int stride, int frames, int pitch, int relu,
                                                    double* __restrict__ stats) {
  __shared__ double red[64];
  const int b = blockIdx.y, f = blockIdx.x * 128 + threadIdx.x;
  const bool valid = f < frames, inb = f < pitch;
  const float* xb = x + (size_t)b * C * T;
  double s = 0.0, ss = 0.0;
  for (int n = 0; n < N; ++n) {
    float acc = 0.f;
    if (valid)
      for (int c = 0; c < C; ++c) {
        const float* wr = W + ((size_t)n * C + c) * L;
        const float* xc = xb + (size_t)c * T;
        for (int k = 0; k < L; ++k) {
          const int t = f * stride + k - pad_left;
          if (t >= 0 && t < T) acc = fmaf(__ldg(wr + k), __ldg(xc + t), acc);
        }
      }
    if (relu) acc = fmaxf(acc, 0.f);
    if (inb) w[((size_t)b * N + n) * pitch + f] = valid ? acc : 0.f;
    if (valid) { s += acc; ss += (double)acc * acc; }
  }
  if (stats != nullptr) {
    block_sum2_d(s, ss, red);
    if (threadIdx.x == 0) { atomicAdd(&stats[2 * b], s); atomicAdd(&stats[2 * b + 1], ss); }
  }
}

__global__ void __launch_bounds__(128) k_decoder_mc(const float* __restrict__ what, const float* __restrict__ Wd, float* __restrict__ y, int C,
                                                    int N, int frames, int in_pitch, int L, int stride, int crop_left, int T_out) {
  const int bs = blockIdx.z, c = blockIdx.y, t = blockIdx.x * 128 + threadIdx.x;
  if (t >= T_out) return;
  const int tau = t + crop_left;
  int f_hi = tau / stride;
  if (f_hi > frames - 1) f_hi = frames - 1;
  int f_lo = (tau - L + stride) / stride;  // smallest f with tau - f*stride <= L - 1
  if (tau - L + 1 <= 0) f_lo = 0;
  float acc = 0.f;
  for (int f = f_lo; f <= f_hi; ++f) {
    const int k = tau - f * stride;
    if (k < 0 || k >= L) continue;
    const float* wh = what + (size_t)bs * N * in_pitch + f;
    const float* wd = Wd + (size_t)c * L + k;
    for (int n = 0; n < N; ++n) acc = fmaf(__ldg(wh + (size_t)n * in_pitch), __ldg(wd + (size_t)n * C * L), acc);
  }
  y[((size_t)bs * C + c) * T_out + t] = acc;
}

extern "C" int ctn_encoder_mc_fwd(const float* x, const float* enc_w, float* w, int B, int C, int T, int pad_left, int pad_right, int N, int L,
                                  int stride, int relu, int w_pitch, double* stats, ctn_stream_t stream) {
  LaunchScope scope(w);
  if (!x || !enc_w || !w || B <= 0 || C <= 0 || T <= 0 || N <= 0 || L <= 0 || stride <= 0) return CTN_EINVAL;
  const int Tp = T + pad_left + pad_right;
  if (Tp < L || (Tp - L) % stride != 0) return CTN_EINVAL;
  const int frames = (Tp - L) / stride + 1;
  if (w_pitch < frames) return CTN_EALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  k_encoder_mc<<<dim3((w_pitch + 127) / 128, B), 128, 0, st>>>(x, enc_w, w, C, T, pad_left, N, L, stride, frames, w_pitch, relu, stats);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

extern "C" int ctn_decoder_mc_fwd(const float* w_hat, const float* dec_w, float* y, int BS, int C, int N, int frames, int in_pitch, int L,
                                  int stride, int crop_left, int T_out, ctn_stream_t stream) {
  LaunchScope scope(w_hat);
  if (!w_hat || !dec_w || !y || BS <= 0 || C <= 0 || C > 65535 || BS > 65535 || N <= 0 || frames <= 0 || L <= 0 || stride <= 0 ||
      L % stride != 0)
    return CTN_EINVAL;
  if (in_pitch < frames) return CTN_EINVAL;
  const int full = (frames - 1) * stride + L;
  if (crop_left < 0 || T_out <= 0 || crop_left + T_out > full) return CTN_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  k_decoder_mc<<<dim3((T_out + 127) / 128, C, BS), 128, 0, st>>>(w_hat, dec_w, y, C, N, frames, in_pitch, L, stride, crop_left, T_out);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}
