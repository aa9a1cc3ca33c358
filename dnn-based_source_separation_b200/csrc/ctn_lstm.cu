// Bidirectional LSTM recurrence + output projection of a dual-path block (BASELINE cfg4) on tcgen05.
// Reference: src/models/dprnn.py:82-90 / 134-142 (x -> nn.LSTM(bidirectional, batch_first) -> nn.Linear(2H, F)); the recurrence
// itself is torch.nn.LSTM: gates (i, f, g, o) = W_ih x_t + b_ih + W_hh h_{t-1} + b_hh, c_t = f c_{t-1} + i g, h_t = o tanh(c_t).
//
// One CTA = 128 sequences (TMEM lanes) of ONE direction, all T steps.  Per step the pre-activations are ONE contraction
//   [x_t | h_{t-1}] (128 x (F + H))  x  [W_ih | W_hh]^T ((F + H) x 4H)
// run as "3xFP16" (hi/lo fp16 pieces, fp32 accumulate in TMEM): gate columns are reordered unit-major (4 gates of a hidden unit
// adjacent) and cut into chunks of 32 units = 128 columns, so that the epilogue of chunk c (sigmoid / tanh, cell update, h_t) runs
// while the tensor core works on chunk c + 1.  Operand placement:
//   * h_{t-1}: in TENSOR MEMORY (tcgen05.mma "ts" form).  The epilogue thread that owns a sequence (= TMEM lane) writes h_t's
//     fp16 hi / lo pieces straight into the A-operand columns with tcgen05.st: h never touches shared or global memory on its
//     way back into the recurrence.  Two h buffers (h_t is produced while later chunks still read h_{t-1}).
//   * x_t: shared memory (K-major SWIZZLE_64B), written by 4 producer warps one step ahead of the recurrence.
//   * weights: pre-split / pre-swizzled 16 KB stage images ([128 columns x 32 k] hi + lo), streamed from L2 through a ring of
//     shared-memory stages by bulk async copies (the whole [W_ih | W_hh | W_fc] set is 442 KB -- more than an SM holds).
//   * the 2H -> F projection of the block (nn.Linear after the LSTM) rides along: one more chunk per step, h_{t-1} (still in
//     TMEM) x W_fc[:, dir*H:(dir+1)*H]^T, so the (NSEQ, T, 2H) LSTM output is never materialised; each direction stores its
//     partial projection (NSEQ, T, F) and the gLN + residual kernel adds the two and the bias.
// TMEM columns: [0,256) two 128-column accumulators, [256,512) two h buffers (hi at +0, lo at +64 of each).
// Warp roles: 0-7 epilogue (warp & 3 = lane quarter, warp >> 2 = column half), 8 TMEM alloc + MMA issuer, 9 weight loader,
// 12-15 x producers.  The launch gives every thread 128 registers; the warpgroups then trade them (setmaxnreg): the epilogue,
// which keeps the cell state of 64 hidden units per thread in registers, runs with 176.
#include "ctn_internal.h"
#include "ctn_umma_ptx.cuh"

namespace {

constexpr int LM = 128;               // sequences per CTA
constexpr int SLAB_BYTES = 16384;     // one weight slab image: [hi 128 columns x 64 B][lo 128 x 64 B] = 32 k of a 128-column chunk
constexpr int STAGE_BYTES = 2 * SLAB_BYTES;  // a ring stage = two consecutive slabs behind one barrier
constexpr int MAX_ST = 6;
constexpr int PSTAGE_BYTES = 32768;   // projection store staging: 8 epilogue warps x 4 KB
constexpr int LSTM_THREADS = 512;     // 4 warpgroups: 0-3, 4-7 epilogue | 8 MMA, 9 loader, 10-11 idle | 12-15 x producers
constexpr int REGS_EPI = 176, REGS_CTRL = 56, REGS_PROD = 104;  // setmaxnreg budget: 128 * (2*176 + 56 + 104) = 65536
constexpr int HDR_BYTES = 1024;

struct LstmScales {                   // one per direction, written by k_lstm_scales
  float x_mul;                        // x operand = x * x_mul            (|.| < 2^14)
  float inv_g;                        // pre-activation = acc * inv_g + bias
  float inv_p;                        // projection = acc * inv_p
  float w_ih_mul, w_hh_mul, w_p_mul;  // weight images = W * mul          (|.| < 2^14)
  float pad[2];
};

struct LstmHdr {
  uint64_t bfull[MAX_ST], bempty[MAX_ST];
  uint64_t accfull[2], accempty[2];
  uint64_t hfull[2];
  uint64_t xfull, xempty;
  uint32_t tmem_base;
};
static_assert(sizeof(LstmHdr) <= HDR_BYTES, "header");

struct LstmArgs {
  const float* z;        // (NSEQ, T, F)
  float* P;              // (2, NSEQ, T, Fo) or null
  float* hout;           // (NSEQ, T, 2H) or null
  const uint8_t* img;    // [2][n_imgs][SLAB_BYTES]
  const float* bias;     // [2][4H], chunk-column order, pre-multiplied by -log2(e) (-2 log2(e) for the g gate)
  const LstmScales* sc;  // [2]
  int NSEQ, T, Fo, n_imgs, n_st, has_proj;
  uint32_t dbg;          // CTN_LSTM_DBG (timing experiments only): 1 no cell math, 2 no MMAs, 4 no weight copies, 8 no x loads
};

__device__ __forceinline__ float ex2f_(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcpf_(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}


// timeline probe (CTN_LSTM_DBG bit 16): cycle stamps of CTA (0,0), steps [100,104): [step][role: 0 issuer, 1 epilogue warp 0][chunk 0..4][4]
__device__ unsigned long long g_lstm_tl[4 * 2 * 5 * 4];
__device__ __forceinline__ void tl_mark(bool on, int t, int role, int c, int k) {
  if (on && t >= 100 && t < 104) g_lstm_tl[(((t - 100) * 2 + role) * 5 + c) * 4 + k] = clock64();
}

template <int N>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// One LSTM cell update.  Inputs are the ex2 ARGUMENTS of the four gates, xi = -log2(e) a_i, xf, xo likewise, xg = -2 log2(e) a_g
// (the scale and the bias are folded into one FFMA by the caller), so that E = 2^x = e^-a (e^-2a for g):
//   sigmoid(a) = 1 / (1 + E),  tanh(a) = (1 - E) / (1 + E).
// f, i*g share ONE reciprocal, o*tanh(c) another: 5 ex2 + 2 rcp per unit (the MUFU pipe, 16 lanes/clk/SM, is what bounds the
// epilogue).  Arguments are capped where the function has saturated in fp32 (E <= e^20 for the sigmoids, e^30 for tanh) so that
// the products of denominators stay finite (< 2.4e30).
__device__ __forceinline__ void lstm_cell(float xi, float xf, float xg, float xo, float& c, float& h) {
  constexpr float CAP_S = 28.853901f, CAP_T = 43.280851f;  // 20 log2(e), 30 log2(e)
  const float Ei = ex2f_(fminf(xi, CAP_S)), Ef = ex2f_(fminf(xf, CAP_S)), Eg = ex2f_(fminf(xg, CAP_T)), Eo = ex2f_(fminf(xo, CAP_S));
  const float pf = 1.f + Ef, pig = (1.f + Ei) * (1.f + Eg);
  const float r = rcpf_(pig * pf);
  c = fmaf(r * pig, c, (1.f - Eg) * (r * pf));
  const float Ec = ex2f_(fminf(c * -2.8853901f, CAP_T));
  h = (1.f - Ec) * rcpf_((1.f + Eo) * (1.f + Ec));
}

// NCH = H / 32 gate chunks, KSX = F / 32 input slabs
template <int NCH, int KSX>
__global__ void __launch_bounds__(LSTM_THREADS, 1) k_bilstm(const LstmArgs g) {
  constexpr int H = 32 * NCH, F = 32 * KSX, KSH = NCH;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  LstmHdr* hdr = reinterpret_cast<LstmHdr*>(smem);
  float* s_bias = reinterpret_cast<float*>(smem + HDR_BYTES);            // 4H floats (<= 2 KB)
  constexpr uint32_t XS_OFF = HDR_BYTES + 2048;                          // x operand: [hi KSX slabs][lo KSX slabs] of 8 KB
  constexpr uint32_t PST_OFF = XS_OFF + 2 * KSX * 8192;                  // projection store staging
  constexpr uint32_t RING_OFF = PST_OFF + PSTAGE_BYTES;
  const uint32_t xs0 = base + XS_OFF, ring0 = base + RING_OFF;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int dir = blockIdx.y, seq0 = blockIdx.x * LM;
  const int T = g.T;
  const bool proj = g.has_proj != 0;
  const LstmScales sc = g.sc[dir];

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.n_st; ++s) {
      ptx::mbar_init(ptx::smem_u32(&hdr->bfull[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->bempty[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(ptx::smem_u32(&hdr->accfull[i]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->accempty[i]), 8);
      ptx::mbar_init(ptx::smem_u32(&hdr->hfull[i]), 8 * NCH);
    }
    ptx::mbar_init(ptx::smem_u32(&hdr->xfull), 4);
    ptx::mbar_init(ptx::smem_u32(&hdr->xempty), 1);
    ptx::fence_mbar_init();
  }
  if (warp == 8) ptx::tmem_alloc(ptx::smem_u32(&hdr->tmem_base), 512);
  for (int i = threadIdx.x; i < 4 * H; i += blockDim.x) s_bias[i] = __ldg(g.bias + (size_t)dir * 4 * H + i);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = hdr->tmem_base;
  const uint32_t tm_h0 = tmem + 256u;  // h buffer b: tm_h0 + b * 128 (hi), + 64 (lo)
  if (warp < 8) {
    // h_{-1} = 0 lives in buffer 1: every epilogue warp clears its lane quarter / column half
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    for (int cc = 0; cc < 64; cc += 8) ptx::tmem_st8(tm_h0 + 128u + lane_off + (uint32_t)((warp >> 2) * 64 + cc), zero);
    ptx::tmem_st_wait();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();

  if (warp >= 8 && warp < 12) reg_dec<REGS_CTRL>();
  if (warp == 9) {
    // ===================================== WEIGHT LOADER ====================================================
    // a ring stage holds TWO consecutive slabs of a sequence (gate slabs of a step / projection slabs of a step), one barrier
    if (ptx::elect_one()) {
      const uint8_t* img = g.img + (size_t)dir * g.n_imgs * SLAB_BYTES;
      int s = 0;
      uint32_t ph = 0;
      auto load_seq = [&](int first, int count, uint32_t bytes) {
        for (int i = 0; i < count; i += 2) {
          const int n = count - i < 2 ? count - i : 2;
          ptx::mbar_wait(ptx::smem_u32(&hdr->bempty[s]), ph ^ 1u);
          const uint32_t fb = ptx::smem_u32(&hdr->bfull[s]);
          ptx::mbar_arrive_expect_tx(fb, bytes * n);
          for (int j = 0; j < n; ++j) {
            if (!(g.dbg & 4u))
              ptx::bulk_g2s(ring0 + (uint32_t)s * STAGE_BYTES + (uint32_t)j * SLAB_BYTES, img + (size_t)(first + i + j) * SLAB_BYTES, bytes, fb);
            else
              asm volatile("mbarrier.complete_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(fb), "r"(bytes) : "memory");
          }
          if (++s == g.n_st) { s = 0; ph ^= 1u; }
        }
      };
      for (int t = 0; t <= T; ++t) {
        if (t < T) load_seq(0, NCH * (KSX + KSH), SLAB_BYTES);
        if (proj && t >= 1) load_seq(NCH * (KSX + KSH), KSH, (uint32_t)g.Fo * 128u);
      }
    }
    __syncwarp();
  } else if (warp == 8) {
    // ===================================== MMA ISSUER =======================================================
    // ONE thread runs the whole loop (waits included): nothing but the barrier waits stands between two groups of MMAs
    if (ptx::elect_one()) {
      const bool do_mma = !(g.dbg & 2u);
      const bool tl = (g.dbg & 16u) && blockIdx.x == 0 && blockIdx.y == 0;
      const uint64_t d_t = ptx::make_smem_desc(0, 16u, 512u, 4u);  // K-major SWIZZLE_64B rows of 32 k (x operand and weights)
      const uint32_t idesc_g = ptx::make_idesc_f16(LM, 128, 0, 0), idesc_p = ptx::make_idesc_f16(LM, g.Fo, 0, 0);
      int s = 0, gidx = 0;
      uint32_t ph = 0;
      // slab i of a sequence of `count`: wait for its stage on the first slab, hand the stage back after the last
      auto acquire = [&](int i) -> uint32_t {
        if (!(i & 1)) {
          ptx::mbar_wait(ptx::smem_u32(&hdr->bfull[s]), ph);
          ptx::tc_fence_after();
        }
        return (ring0 + (uint32_t)s * STAGE_BYTES + (uint32_t)(i & 1) * SLAB_BYTES) >> 4;
      };
      auto release = [&](int i, int count) {
        if ((i & 1) || i == count - 1) {
          ptx::mma_commit(ptx::smem_u32(&hdr->bempty[s]));
          if (++s == g.n_st) { s = 0; ph ^= 1u; }
        }
      };
      for (int t = 0; t <= T; ++t) {
        const uint32_t h_prev = tm_h0 + (uint32_t)((t + 1) & 1) * 128u;  // buffer holding h_{t-1}
        if (t < T) {
#pragma unroll 1
          for (int c = 0; c < NCH; ++c) {
            const int slot = gidx & 1;
            ptx::mbar_wait(ptx::smem_u32(&hdr->accempty[slot]), ((uint32_t)(gidx >> 1) & 1u) ^ 1u);
            if (c == 0) ptx::mbar_wait(ptx::smem_u32(&hdr->xfull), (uint32_t)t & 1u);
            ptx::tc_fence_after();
            tl_mark(tl, t, 0, c, 0);
            const uint32_t d_tmem = tmem + (uint32_t)slot * 128u;
#pragma unroll 1
            for (int k = 0; k < KSX; ++k) {
              const int i = c * (KSX + KSH) + k;
              const uint32_t w_hi = acquire(i), w_lo = w_hi + (8192u >> 4);
              const uint32_t a_hi = (xs0 + (uint32_t)k * 8192u) >> 4, a_lo = a_hi + ((uint32_t)KSX * 8192u >> 4);
#pragma unroll
              for (int kk = 0; kk < 2; ++kk) {
                if (!do_mma) break;
                ptx::mma_f16(d_tmem, d_t | (uint64_t)(a_hi + kk * 2), d_t | (uint64_t)(w_hi + kk * 2), idesc_g, (k | kk) ? 1u : 0u);
                ptx::mma_f16(d_tmem, d_t | (uint64_t)(a_lo + kk * 2), d_t | (uint64_t)(w_hi + kk * 2), idesc_g, 1u);
                ptx::mma_f16(d_tmem, d_t | (uint64_t)(a_hi + kk * 2), d_t | (uint64_t)(w_lo + kk * 2), idesc_g, 1u);
              }
              release(i, NCH * (KSX + KSH));
              if (c == NCH - 1 && k == KSX - 1) ptx::mma_commit(ptx::smem_u32(&hdr->xempty));  // x_t has been consumed
            }
            tl_mark(tl, t, 0, c, 1);
            if (c == 0 && t > 0) {
              ptx::mbar_wait(ptx::smem_u32(&hdr->hfull[(t + 1) & 1]), (uint32_t)((t - 1) >> 1) & 1u);
              ptx::tc_fence_after();
            }
            tl_mark(tl, t, 0, c, 2);
#pragma unroll 1
            for (int k = 0; k < KSH; ++k) {
              const int i = c * (KSX + KSH) + KSX + k;
              const uint32_t w_hi = acquire(i), w_lo = w_hi + (8192u >> 4);
#pragma unroll
              for (int kk = 0; kk < 2; ++kk) {
                if (!do_mma) break;
                const uint32_t a_hi = h_prev + (uint32_t)(k * 2 + kk) * 8u, a_lo = a_hi + 64u;
                ptx::mma_f16_ts(d_tmem, a_hi, d_t | (uint64_t)(w_hi + kk * 2), idesc_g, 1u);
                ptx::mma_f16_ts(d_tmem, a_lo, d_t | (uint64_t)(w_hi + kk * 2), idesc_g, 1u);
                ptx::mma_f16_ts(d_tmem, a_hi, d_t | (uint64_t)(w_lo + kk * 2), idesc_g, 1u);
              }
              release(i, NCH * (KSX + KSH));
            }
            ptx::mma_commit(ptx::smem_u32(&hdr->accfull[slot]));
            tl_mark(tl, t, 0, c, 3);
            ++gidx;
          }
        }
        if (proj && t >= 1) {
          const int slot = gidx & 1;
          ptx::mbar_wait(ptx::smem_u32(&hdr->accempty[slot]), ((uint32_t)(gidx >> 1) & 1u) ^ 1u);
          if (t == T) ptx::mbar_wait(ptx::smem_u32(&hdr->hfull[(t + 1) & 1]), (uint32_t)((t - 1) >> 1) & 1u);
          ptx::tc_fence_after();
          tl_mark(tl, t, 0, 4, 0);
          const uint32_t d_tmem = tmem + (uint32_t)slot * 128u;
          const uint32_t lo_off = ((uint32_t)g.Fo * 64u) >> 4;
#pragma unroll 1
          for (int k = 0; k < KSH; ++k) {
            const uint32_t w_hi = acquire(k), w_lo = w_hi + lo_off;
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              if (!do_mma) break;
              const uint32_t a_hi = h_prev + (uint32_t)(k * 2 + kk) * 8u, a_lo = a_hi + 64u;
              ptx::mma_f16_ts(d_tmem, a_hi, d_t | (uint64_t)(w_hi + kk * 2), idesc_p, (k | kk) ? 1u : 0u);
              ptx::mma_f16_ts(d_tmem, a_lo, d_t | (uint64_t)(w_hi + kk * 2), idesc_p, 1u);
              ptx::mma_f16_ts(d_tmem, a_hi, d_t | (uint64_t)(w_lo + kk * 2), idesc_p, 1u);
            }
            release(k, KSH);
          }
          ptx::mma_commit(ptx::smem_u32(&hdr->accfull[slot]));
          tl_mark(tl, t, 0, 4, 3);
          ++gidx;
        }
      }
    }
    __syncwarp();
  } else if (warp >= 12) {
    // ===================================== x PRODUCERS ======================================================
    // thread = one sequence: x_t (F floats, contiguous) -> scaled fp16 hi / lo pieces -> K-major SWIZZLE_64B slabs
    reg_dec<REGS_PROD>();
    const int r = (warp - 12) * 32 + lane, seq = seq0 + r;
    const bool valid = seq < g.NSEQ;
    const float4* zrow = reinterpret_cast<const float4*>(g.z + (size_t)(valid ? seq : 0) * T * F);
    uint8_t* xs = smem + XS_OFF;
    const uint32_t row_off = (uint32_t)(r >> 3) * 512u + (uint32_t)(r & 7) * 64u, sw = (uint32_t)(r >> 1) & 3u;
    float4 v[F / 4];
    auto fetch = [&](int t) {
      const int ti = dir ? T - 1 - t : t;
#pragma unroll
      for (int i = 0; i < F / 4; ++i)
        v[i] = (valid && !(g.dbg & 8u)) ? __ldg(zrow + (size_t)ti * (F / 4) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    fetch(0);
    for (int t = 0; t < T; ++t) {
      if (t > 0) ptx::mbar_wait(ptx::smem_u32(&hdr->xempty), (uint32_t)(t - 1) & 1u);
#pragma unroll
      for (int k = 0; k < KSX; ++k) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {  // 16-byte chunk j of the slab row: k-elements 8j .. 8j+7
          const float4 a = v[k * 8 + j * 2], b = v[k * 8 + j * 2 + 1];
          uint4 hi, lo;
          ptx::split_f16x2(a.x * sc.x_mul, a.y * sc.x_mul, hi.x, lo.x);
          ptx::split_f16x2(a.z * sc.x_mul, a.w * sc.x_mul, hi.y, lo.y);
          ptx::split_f16x2(b.x * sc.x_mul, b.y * sc.x_mul, hi.z, lo.z);
          ptx::split_f16x2(b.z * sc.x_mul, b.w * sc.x_mul, hi.w, lo.w);
          const uint32_t off = (uint32_t)k * 8192u + row_off + (((uint32_t)j ^ sw) << 4);
          *reinterpret_cast<uint4*>(xs + off) = hi;
          *reinterpret_cast<uint4*>(xs + (uint32_t)KSX * 8192u + off) = lo;
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->xfull));
      if (t + 1 < T) fetch(t + 1);
    }
  } else if (warp < 8) {
    // ===================================== EPILOGUE =========================================================
    reg_inc<REGS_EPI>();
    const int q = warp & 3, e = warp >> 2;
    const float sg = -1.4426950408889634f * sc.inv_g, sg2 = 2.f * sg;  // acc -> ex2 argument (bias table is pre-scaled alike)
    const bool tl = (g.dbg & 16u) && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0;
    const int r = q * 32 + lane, seq = seq0 + r;
    const bool valid = seq < g.NSEQ;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    float cst[NCH][16];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int u = 0; u < 16; ++u) cst[c][u] = 0.f;
    int gidx = 0;
    for (int t = 0; t <= T; ++t) {
      if (t < T) {
        const int ti = dir ? T - 1 - t : t;
        const uint32_t h_cur = tm_h0 + (uint32_t)(t & 1) * 128u;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int slot = gidx & 1;
          ptx::mbar_wait(ptx::smem_u32(&hdr->accfull[slot]), (uint32_t)(gidx >> 1) & 1u);
          ptx::tc_fence_after();
          tl_mark(tl, t, 1, c, 0);
          float hv[16];
          uint32_t a0[32], a1[32];
          ptx::tmem_ld32(tmem + lane_off + (uint32_t)(slot * 128 + e * 64), a0);
          ptx::tmem_ld32(tmem + lane_off + (uint32_t)(slot * 128 + e * 64 + 32), a1);
          ptx::tmem_ld_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->accempty[slot]));  // the accumulator is in registers: slot free
          tl_mark(tl, t, 1, c, 1);
          const float4* bp = reinterpret_cast<const float4*>(s_bias + c * 128 + e * 64);
          if (g.dbg & 1u) {
#pragma unroll
            for (int u = 0; u < 16; ++u) hv[u] = 1e-6f * __uint_as_float(u < 8 ? a0[4 * u] : a1[4 * (u - 8)]);
          } else {
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float4 bb = bp[u];
            lstm_cell(fmaf(__uint_as_float(a0[4 * u]), sg, bb.x), fmaf(__uint_as_float(a0[4 * u + 1]), sg, bb.y),
                      fmaf(__uint_as_float(a0[4 * u + 2]), sg2, bb.z), fmaf(__uint_as_float(a0[4 * u + 3]), sg, bb.w), cst[c][u], hv[u]);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float4 bb = bp[8 + u];
            lstm_cell(fmaf(__uint_as_float(a1[4 * u]), sg, bb.x), fmaf(__uint_as_float(a1[4 * u + 1]), sg, bb.y),
                      fmaf(__uint_as_float(a1[4 * u + 2]), sg2, bb.z), fmaf(__uint_as_float(a1[4 * u + 3]), sg, bb.w), cst[c][8 + u],
                      hv[8 + u]);
          }
          }
          tl_mark(tl, t, 1, c, 2);
          // h_t pieces for the next step: units 32c + 16e + [0,16) -> 8 packed columns of the hi image, 8 of the lo image
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) ptx::split_f16x2(hv[2 * i] * 16384.f, hv[2 * i + 1] * 16384.f, hi[i], lo[i]);
          ptx::tmem_st8(h_cur + lane_off + (uint32_t)(c * 16 + e * 8), hi);
          ptx::tmem_st8(h_cur + lane_off + 64u + (uint32_t)(c * 16 + e * 8), lo);
          ptx::tmem_st_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->hfull[t & 1]));
          tl_mark(tl, t, 1, c, 3);
          if (g.hout && valid) {
            float4* dst = reinterpret_cast<float4*>(g.hout + ((size_t)seq * T + ti) * (2 * H) + dir * H + c * 32 + e * 16);
#pragma unroll
            for (int i = 0; i < 4; ++i) dst[i] = make_float4(hv[4 * i], hv[4 * i + 1], hv[4 * i + 2], hv[4 * i + 3]);
          }
          ++gidx;
        }
      }
      if (proj && t >= 1) {
        const int tp = dir ? T - t : t - 1;  // time index of h_{t-1}
        const int slot = gidx & 1;
        ptx::mbar_wait(ptx::smem_u32(&hdr->accfull[slot]), (uint32_t)(gidx >> 1) & 1u);
        ptx::tc_fence_after();
        tl_mark(tl, t, 1, 4, 0);
        // this warp's 32 rows x (Fo/2) columns, in pieces of 32 (or 16) columns: registers (thread = row) -> swizzled shared
        // staging -> global with 8 (4) consecutive lanes covering one row's 128 (64) contiguous bytes
        const int half_cols = g.Fo >> 1;
        float4* pst = reinterpret_cast<float4*>(smem + PST_OFF + warp * 4096);
        const size_t row_base = ((size_t)dir * g.NSEQ + seq0 + q * 32) * T + tp;  // + row * T
        for (int c0 = 0; c0 < half_cols; c0 += 32) {
          const int w = half_cols - c0 >= 32 ? 32 : 16;
          uint32_t a[32];
          if (w == 32) ptx::tmem_ld32(tmem + lane_off + (uint32_t)(slot * 128 + e * half_cols + c0), a);
          else ptx::tmem_ld16(tmem + lane_off + (uint32_t)(slot * 128 + e * half_cols + c0), reinterpret_cast<uint32_t(&)[16]>(a));
          ptx::tmem_ld_wait();
          if (c0 + 32 >= half_cols) {  // last piece: the accumulator is in registers
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->accempty[slot]));
          }
          if (w == 32) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              pst[lane * 8 + (i ^ (lane & 7))] = make_float4(__uint_as_float(a[4 * i]) * sc.inv_p, __uint_as_float(a[4 * i + 1]) * sc.inv_p,
                                                             __uint_as_float(a[4 * i + 2]) * sc.inv_p, __uint_as_float(a[4 * i + 3]) * sc.inv_p);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int row = j * 4 + (lane >> 3), qq = lane & 7;
              const float4 v = pst[row * 8 + (qq ^ (row & 7))];
              if (seq0 + q * 32 + row < g.NSEQ)
                *reinterpret_cast<float4*>(g.P + (row_base + (size_t)row * T) * g.Fo + e * half_cols + c0 + qq * 4) = v;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              pst[lane * 4 + (i ^ (lane & 3))] = make_float4(__uint_as_float(a[4 * i]) * sc.inv_p, __uint_as_float(a[4 * i + 1]) * sc.inv_p,
                                                             __uint_as_float(a[4 * i + 2]) * sc.inv_p, __uint_as_float(a[4 * i + 3]) * sc.inv_p);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int row = j * 8 + (lane >> 2), qq = lane & 3;
              const float4 v = pst[row * 4 + (qq ^ (row & 3))];
              if (seq0 + q * 32 + row < g.NSEQ)
                *reinterpret_cast<float4*>(g.P + (row_base + (size_t)row * T) * g.Fo + e * half_cols + c0 + qq * 4) = v;
            }
          }
          __syncwarp();
        }
        tl_mark(tl, t, 1, 4, 3);
        ++gidx;
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (warp == 8) ptx::tmem_dealloc(tmem, 512);
}

// =====================================================================================================================
// 2-CTA form.  A cluster of two CTAs shares the 128 sequences of one direction: CTA `rank` owns hidden units
// [rank H/2, (rank+1) H/2) -- their gate columns (CH = H/64 chunks), their cell state, and half of the projection's output
// features -- so both the tensor-core time and the sigmoid/tanh time of a step halve, and twice as many SMs work on the
// (small) cfg4 batch.  Each step the two CTAs exchange their halves of h_t:
//   * own half: TMEM A operand, written by the epilogue with tcgen05.st as in the 1-CTA kernel;
//   * the SAME pieces are also stored to a shared-memory staging slab in operand layout (K-major SWIZZLE_64B, 128 x 32 k,
//     hi + lo = 16 KB per chunk) and a sender warp pushes each slab into the peer's shared memory with one bulk
//     shared::cta -> shared::cluster copy that completes on the PEER's mbarrier (complete_tx): the peer's MMAs read it as a
//     shared-memory A operand, async proxy end to end.
//   * buffer reuse: the peer's in-buffer b is overwritten every other step; the reader side says when it is done with it by a
//     tcgen05.commit multicast onto the sender's `pfree[b]` barrier (arrives when the reading MMAs have completed).
// x_t now lives in TMEM too (the x producers own one lane each): shared memory holds only weights (ring), the two exchange
// buffers and the store staging.  K order of a gate chunk: [x | own h | peer h] -- the peer's half arrives last.
// TMEM columns: [0,256) accumulators, [256,384) own-h buffers (64 each: hi +0, lo +32), [384,512) x (hi +0, lo +64).
constexpr int PAIR_MAX_ST = 8;
struct PairHdr {
  uint64_t bfull[PAIR_MAX_ST], bempty[PAIR_MAX_ST];
  uint64_t accfull[2], accempty[2];
  uint64_t hfull[2];
  uint64_t xfull, xempty;
  uint64_t outfull[2][2];  // [buffer][piece]: the 8 epilogue warps -> sender warp
  uint64_t pin[2][2];      // [buffer][piece]: the peer's piece has landed in my in-buffer (transaction bytes)
  uint64_t pfree[2];       // the PEER no longer reads ITS in-buffer b (arrives from the peer's tcgen05.commit)
  uint32_t tmem_base;
};
static_assert(sizeof(PairHdr) <= HDR_BYTES, "header");

template <int NCH, int KSX>
__global__ void __launch_bounds__(LSTM_THREADS, 1) k_bilstm_pair(const LstmArgs g) {
  constexpr int CH = NCH / 2, H = 32 * NCH, HL = 32 * CH, F = 32 * KSX, GSL = KSX + NCH;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  PairHdr* hdr = reinterpret_cast<PairHdr*>(smem);
  float* s_bias = reinterpret_cast<float*>(smem + HDR_BYTES);  // 4 * HL floats (<= 1 KB)
  constexpr uint32_t PST_OFF = 2 * HDR_BYTES;
  const uint32_t out_off = PST_OFF + 256u * (uint32_t)g.Fo;     // store staging: 8 warps x 32 rows x Fo/4 floats
  const uint32_t in_off = out_off + 2u * CH * SLAB_BYTES, ring_off = in_off + 2u * CH * SLAB_BYTES;
  const uint32_t out0 = base + out_off, in0 = base + in_off, ring0 = base + ring_off;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)ptx::cluster_ctarank(), peer = rank ^ 1;
  const int dir = blockIdx.y, seq0 = (int)(blockIdx.x >> 1) * LM;
  const int T = g.T;
  const bool proj = g.has_proj != 0;
  const LstmScales sc = g.sc[dir];

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.n_st; ++s) {
      ptx::mbar_init(ptx::smem_u32(&hdr->bfull[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->bempty[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(ptx::smem_u32(&hdr->accfull[i]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->accempty[i]), 8);
      ptx::mbar_init(ptx::smem_u32(&hdr->hfull[i]), 8 * CH);
      ptx::mbar_init(ptx::smem_u32(&hdr->pfree[i]), 1);
      for (int c = 0; c < 2; ++c) {
        ptx::mbar_init(ptx::smem_u32(&hdr->outfull[i][c]), 8);
        ptx::mbar_init(ptx::smem_u32(&hdr->pin[i][c]), 1);
      }
    }
    ptx::mbar_init(ptx::smem_u32(&hdr->xfull), 4);
    ptx::mbar_init(ptx::smem_u32(&hdr->xempty), 1);
    ptx::fence_mbar_init();
  }
  if (warp == 8) ptx::tmem_alloc(ptx::smem_u32(&hdr->tmem_base), 512);
  for (int i = threadIdx.x; i < 4 * HL; i += blockDim.x) s_bias[i] = __ldg(g.bias + (size_t)(dir * 2 + rank) * 4 * HL + i);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  ptx::cluster_sync_all();  // both CTAs' barriers exist before any remote copy / arrive / commit
  const uint32_t tmem = hdr->tmem_base;
  const uint32_t tm_h0 = tmem + 256u, tm_x = tmem + 384u;

  if (warp >= 8 && warp < 12) reg_dec<REGS_CTRL>();
  if (warp == 9) {
    // ===================================== WEIGHT LOADER ====================================================
    if (ptx::elect_one()) {
      const uint8_t* img = g.img + (size_t)(dir * 2 + rank) * g.n_imgs * SLAB_BYTES;
      int s = 0;
      uint32_t ph = 0;
      auto load = [&](int idx, uint32_t bytes) {
        ptx::mbar_wait(ptx::smem_u32(&hdr->bempty[s]), ph ^ 1u);
        const uint32_t fb = ptx::smem_u32(&hdr->bfull[s]);
        ptx::mbar_arrive_expect_tx(fb, bytes);
        if (!(g.dbg & 4u)) ptx::bulk_g2s(ring0 + (uint32_t)s * SLAB_BYTES, img + (size_t)idx * SLAB_BYTES, bytes, fb);
        else asm volatile("mbarrier.complete_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(fb), "r"(bytes) : "memory");
        if (++s == g.n_st) { s = 0; ph ^= 1u; }
      };
      for (int t = 0; t <= T; ++t) {
        if (t < T)
          for (int c = 0; c < CH; ++c)
            for (int k = 0; k < (t == 0 ? KSX : GSL); ++k) load(c * GSL + k, SLAB_BYTES);  // h_{-1} = 0: no h slabs at t = 0
        if (proj && t >= 1)
          for (int k = 0; k < NCH; ++k) load(CH * GSL + k, (uint32_t)g.Fo * 64u);
      }
    }
    __syncwarp();
  } else if (warp == 8) {
    // ===================================== MMA ISSUER =======================================================
    if (ptx::elect_one()) {
      const bool do_mma = !(g.dbg & 2u);
      const bool tl = (g.dbg & 16u) && blockIdx.x == 0 && blockIdx.y == 0;
      const uint64_t d_t = ptx::make_smem_desc(0, 16u, 512u, 4u);
      const uint32_t idesc_g = ptx::make_idesc_f16(LM, 128, 0, 0), idesc_p = ptx::make_idesc_f16(LM, g.Fo >> 1, 0, 0);
      for (int b = 0; b < 2; ++b)
        for (int c = 0; c < CH; ++c) ptx::mbar_arrive_expect_tx(ptx::smem_u32(&hdr->pin[b][c]), SLAB_BYTES);
      int s = 0, gidx = 0;
      uint32_t ph = 0;
      auto acquire = [&]() -> uint32_t {
        ptx::mbar_wait(ptx::smem_u32(&hdr->bfull[s]), ph);
        ptx::tc_fence_after();
        return (ring0 + (uint32_t)s * SLAB_BYTES) >> 4;
      };
      auto release = [&]() {
        ptx::mma_commit(ptx::smem_u32(&hdr->bempty[s]));
        if (++s == g.n_st) { s = 0; ph ^= 1u; }
      };
      // three passes of one 32-k slab: A pieces either in TMEM (taddr of the hi piece, lo `a_lo_off` columns further) ...
      auto slab_ts = [&](uint32_t d_tmem, uint32_t a_hi0, uint32_t a_lo_off, uint32_t w_hi, uint32_t w_lo, uint32_t idesc, bool first) {
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          if (!do_mma) break;
          const uint32_t a_hi = a_hi0 + (uint32_t)kk * 8u, a_lo = a_hi + a_lo_off;
          ptx::mma_f16_ts(d_tmem, a_hi, d_t | (uint64_t)(w_hi + kk * 2), idesc, (first && kk == 0) ? 0u : 1u);
          ptx::mma_f16_ts(d_tmem, a_lo, d_t | (uint64_t)(w_hi + kk * 2), idesc, 1u);
          ptx::mma_f16_ts(d_tmem, a_hi, d_t | (uint64_t)(w_lo + kk * 2), idesc, 1u);
        }
      };
      // ... or in shared memory (descriptor address >> 4 of the hi image, lo image 8 KB further)
      auto slab_ss = [&](uint32_t d_tmem, uint32_t a_hi0, uint32_t w_hi, uint32_t w_lo, uint32_t idesc, bool first) {
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          if (!do_mma) break;
          const uint32_t a_hi = a_hi0 + (uint32_t)kk * 2u, a_lo = a_hi + (8192u >> 4);
          ptx::mma_f16(d_tmem, d_t | (uint64_t)a_hi, d_t | (uint64_t)(w_hi + kk * 2), idesc, (first && kk == 0) ? 0u : 1u);
          ptx::mma_f16(d_tmem, d_t | (uint64_t)a_lo, d_t | (uint64_t)(w_hi + kk * 2), idesc, 1u);
          ptx::mma_f16(d_tmem, d_t | (uint64_t)a_hi, d_t | (uint64_t)(w_lo + kk * 2), idesc, 1u);
        }
      };
      for (int t = 0; t <= T; ++t) {
        const int hb = (t + 1) & 1;  // buffer index of h_{t-1}
        const uint32_t h_own = tm_h0 + (uint32_t)hb * 64u, h_peer = (in0 + (uint32_t)hb * CH * SLAB_BYTES) >> 4;
        bool h_ready = false;
        auto need_h = [&]() {
          if (h_ready) return;
          const uint32_t par = (uint32_t)((t - 1) >> 1) & 1u;
          ptx::mbar_wait(ptx::smem_u32(&hdr->hfull[hb]), par);
          for (int c = 0; c < CH; ++c) {
            ptx::mbar_wait_cluster(ptx::smem_u32(&hdr->pin[hb][c]), par);
            ptx::mbar_arrive_expect_tx(ptx::smem_u32(&hdr->pin[hb][c]), SLAB_BYTES);  // arm the next use (h_{t+1})
          }
          ptx::tc_fence_after();
          h_ready = true;
        };
        if (t < T) {
#pragma unroll 1
          for (int c = 0; c < CH; ++c) {
            const int slot = gidx & 1;
            ptx::mbar_wait(ptx::smem_u32(&hdr->accempty[slot]), ((uint32_t)(gidx >> 1) & 1u) ^ 1u);
            if (c == 0) ptx::mbar_wait(ptx::smem_u32(&hdr->xfull), (uint32_t)t & 1u);
            ptx::tc_fence_after();
            tl_mark(tl, t, 0, c, 0);
            const uint32_t d_tmem = tmem + (uint32_t)slot * 128u;
#pragma unroll 1
            for (int k = 0; k < KSX; ++k) {
              const uint32_t w_hi = acquire();
              slab_ts(d_tmem, tm_x + (uint32_t)k * 16u, 64u, w_hi, w_hi + (8192u >> 4), idesc_g, k == 0);
              release();
            }
            if (c == CH - 1) ptx::mma_commit(ptx::smem_u32(&hdr->xempty));  // x_t has been consumed
            tl_mark(tl, t, 0, c, 1);
            if (t > 0) {
              need_h();
              tl_mark(tl, t, 0, c, 2);
#pragma unroll 1
              for (int k = 0; k < CH; ++k) {
                const uint32_t w_hi = acquire();
                slab_ts(d_tmem, h_own + (uint32_t)k * 16u, 32u, w_hi, w_hi + (8192u >> 4), idesc_g, false);
                release();
              }
#pragma unroll 1
              for (int k = 0; k < CH; ++k) {
                const uint32_t w_hi = acquire();
                slab_ss(d_tmem, h_peer + (uint32_t)k * (SLAB_BYTES >> 4), w_hi, w_hi + (8192u >> 4), idesc_g, false);
                release();
              }
            }
            ptx::mma_commit(ptx::smem_u32(&hdr->accfull[slot]));
            tl_mark(tl, t, 0, c, 3);
            ++gidx;
          }
        }
        if (proj && t >= 1) {
          const int slot = gidx & 1;
          ptx::mbar_wait(ptx::smem_u32(&hdr->accempty[slot]), ((uint32_t)(gidx >> 1) & 1u) ^ 1u);
          need_h();
          ptx::tc_fence_after();
          tl_mark(tl, t, 0, 4, 0);
          const uint32_t d_tmem = tmem + (uint32_t)slot * 128u;
          const uint32_t lo_off = ((uint32_t)g.Fo * 32u) >> 4;  // hi image: Fo/2 rows x 64 B
#pragma unroll 1
          for (int k = 0; k < NCH; ++k) {
            const uint32_t w_hi = acquire();
            if (k < CH) slab_ts(d_tmem, h_own + (uint32_t)k * 16u, 32u, w_hi, w_hi + lo_off, idesc_p, k == 0);
            else slab_ss(d_tmem, h_peer + (uint32_t)(k - CH) * (SLAB_BYTES >> 4), w_hi, w_hi + lo_off, idesc_p, false);
            release();
          }
          ptx::mma_commit(ptx::smem_u32(&hdr->accfull[slot]));
          tl_mark(tl, t, 0, 4, 3);
          ++gidx;
        }
        // every MMA that reads in-buffer hb has been issued: when they complete the peer may overwrite it (with h_{t+1})
        if (t >= 1 && t + 1 < T) ptx::mma_commit_multicast(ptx::smem_u32(&hdr->pfree[hb]), (uint16_t)(1u << peer));
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    // ===================================== SENDER ===========================================================
    if (ptx::elect_one()) {
      // h_{T-1} is only read by the final projection: without one nobody waits for it on the other side, and a copy must never be
      // left in flight towards a CTA that may already have exited
      const int t_send = proj ? T : T - 1;
      for (int t = 0; t < t_send; ++t) {
        const int b = t & 1;
        if (t >= 2) ptx::mbar_wait_cluster(ptx::smem_u32(&hdr->pfree[b]), (uint32_t)((t >> 1) - 1) & 1u);
        for (int c = 0; c < CH; ++c) {
          ptx::mbar_wait(ptx::smem_u32(&hdr->outfull[b][c]), (uint32_t)(t >> 1) & 1u);
          const uint32_t off = (uint32_t)(b * CH + c) * SLAB_BYTES;
          ptx::bulk_s2peer(in0 + off, out0 + off, SLAB_BYTES, ptx::smem_u32(&hdr->pin[b][c]), (uint32_t)peer);
        }
      }
    }
    __syncwarp();
  } else if (warp >= 12) {
    // ===================================== x PRODUCERS ======================================================
    // thread = one sequence = one TMEM lane: x_t -> scaled fp16 hi / lo pieces -> tcgen05.st into the x operand columns
    reg_dec<REGS_PROD>();
    const int r = (warp - 12) * 32 + lane, seq = seq0 + r;
    const bool valid = seq < g.NSEQ;
    const float4* zrow = reinterpret_cast<const float4*>(g.z + (size_t)(valid ? seq : 0) * T * F);
    const uint32_t lane_off = (uint32_t)((warp - 12) * 32) << 16;
    float4 v[F / 4];
    auto fetch = [&](int t) {
      const int ti = dir ? T - 1 - t : t;
#pragma unroll
      for (int i = 0; i < F / 4; ++i)
        v[i] = (valid && !(g.dbg & 8u)) ? __ldg(zrow + (size_t)ti * (F / 4) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    fetch(0);
    for (int t = 0; t < T; ++t) {
      if (t > 0) {
        ptx::mbar_wait(ptx::smem_u32(&hdr->xempty), (uint32_t)(t - 1) & 1u);
        ptx::tc_fence_after();
      }
#pragma unroll
      for (int i = 0; i < F / 16; ++i) {  // 16 k-elements = 8 packed columns per store
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 a = v[i * 4 + j];
          ptx::split_f16x2(a.x * sc.x_mul, a.y * sc.x_mul, hi[2 * j], lo[2 * j]);
          ptx::split_f16x2(a.z * sc.x_mul, a.w * sc.x_mul, hi[2 * j + 1], lo[2 * j + 1]);
        }
        ptx::tmem_st8(tm_x + lane_off + (uint32_t)i * 8u, hi);
        ptx::tmem_st8(tm_x + lane_off + 64u + (uint32_t)i * 8u, lo);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->xfull));
      if (t + 1 < T) fetch(t + 1);
    }
  } else if (warp < 8) {
    // ===================================== EPILOGUE =========================================================
    reg_inc<REGS_EPI>();
    const int q = warp & 3, e = warp >> 2;
    const int r = q * 32 + lane, seq = seq0 + r;
    const bool valid = seq < g.NSEQ;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const float sg = -1.4426950408889634f * sc.inv_g, sg2 = 2.f * sg;
    const bool tl = (g.dbg & 16u) && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0;
    const uint32_t st_off = (uint32_t)(r >> 3) * 512u + (uint32_t)(r & 7) * 64u, sw = (uint32_t)(r >> 1) & 3u;
    float cst[CH][16];
#pragma unroll
    for (int c = 0; c < CH; ++c)
#pragma unroll
      for (int u = 0; u < 16; ++u) cst[c][u] = 0.f;
    int gidx = 0;
    for (int t = 0; t <= T; ++t) {
      if (t < T) {
        const int ti = dir ? T - 1 - t : t;
        const int b = t & 1;
        const uint32_t h_cur = tm_h0 + (uint32_t)b * 64u;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          const int slot = gidx & 1;
          ptx::mbar_wait(ptx::smem_u32(&hdr->accfull[slot]), (uint32_t)(gidx >> 1) & 1u);
          ptx::tc_fence_after();
          tl_mark(tl, t, 1, c, 0);
          float hv[16];
          uint32_t a0[32], a1[32];
          ptx::tmem_ld32(tmem + lane_off + (uint32_t)(slot * 128 + e * 64), a0);
          ptx::tmem_ld32(tmem + lane_off + (uint32_t)(slot * 128 + e * 64 + 32), a1);
          ptx::tmem_ld_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->accempty[slot]));
          tl_mark(tl, t, 1, c, 1);
          const float4* bp = reinterpret_cast<const float4*>(s_bias + c * 128 + e * 64);
          if (g.dbg & 1u) {
#pragma unroll
            for (int u = 0; u < 16; ++u) hv[u] = 1e-6f * __uint_as_float(u < 8 ? a0[4 * u] : a1[4 * (u - 8)]);
          } else {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float4 bb = bp[u];
              lstm_cell(fmaf(__uint_as_float(a0[4 * u]), sg, bb.x), fmaf(__uint_as_float(a0[4 * u + 1]), sg, bb.y),
                        fmaf(__uint_as_float(a0[4 * u + 2]), sg2, bb.z), fmaf(__uint_as_float(a0[4 * u + 3]), sg, bb.w), cst[c][u], hv[u]);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float4 bb = bp[8 + u];
              lstm_cell(fmaf(__uint_as_float(a1[4 * u]), sg, bb.x), fmaf(__uint_as_float(a1[4 * u + 1]), sg, bb.y),
                        fmaf(__uint_as_float(a1[4 * u + 2]), sg2, bb.z), fmaf(__uint_as_float(a1[4 * u + 3]), sg, bb.w), cst[c][8 + u],
                        hv[8 + u]);
            }
          }
          tl_mark(tl, t, 1, c, 2);
          // h_t pieces: (1) the peer's copy -- operand-layout staging slab, units 16e + [0,16) of this chunk = 16-byte chunks 2e, 2e+1
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) ptx::split_f16x2(hv[2 * i] * 16384.f, hv[2 * i + 1] * 16384.f, hi[i], lo[i]);
          uint8_t* piece = smem + out_off + (uint32_t)(b * CH + c) * SLAB_BYTES + st_off;
          *reinterpret_cast<uint4*>(piece + (((uint32_t)(2 * e) ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(piece + (((uint32_t)(2 * e + 1) ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
          *reinterpret_cast<uint4*>(piece + 8192 + (((uint32_t)(2 * e) ^ sw) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(piece + 8192 + (((uint32_t)(2 * e + 1) ^ sw) << 4)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
          ptx::fence_proxy_async_smem();
          tl_mark(tl, t, 1, c + 2, 0);
          // (2) my own copy: TMEM A-operand columns of buffer b
          if (!(g.dbg & 32u)) {
            ptx::tmem_st8(h_cur + lane_off + (uint32_t)(c * 16 + e * 8), hi);
            ptx::tmem_st8(h_cur + lane_off + 32u + (uint32_t)(c * 16 + e * 8), lo);
          }
          tl_mark(tl, t, 1, c + 2, 1);
          ptx::tmem_st_wait();
          tl_mark(tl, t, 1, c + 2, 2);
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            ptx::mbar_arrive(ptx::smem_u32(&hdr->outfull[b][c]));
            ptx::mbar_arrive(ptx::smem_u32(&hdr->hfull[b]));
          }
          tl_mark(tl, t, 1, c, 3);
          if (g.hout && valid) {
            float4* dst = reinterpret_cast<float4*>(g.hout + ((size_t)seq * T + ti) * (2 * H) + dir * H + (rank * CH + c) * 32 + e * 16);
#pragma unroll
            for (int i = 0; i < 4; ++i) dst[i] = make_float4(hv[4 * i], hv[4 * i + 1], hv[4 * i + 2], hv[4 * i + 3]);
          }
          ++gidx;
        }
      }
      if (proj && t >= 1) {
        const int tp = dir ? T - t : t - 1;  // time index of h_{t-1}
        const int slot = gidx & 1;
        ptx::mbar_wait(ptx::smem_u32(&hdr->accfull[slot]), (uint32_t)(gidx >> 1) & 1u);
        ptx::tc_fence_after();
        tl_mark(tl, t, 1, 4, 0);
        // this CTA's Fo/2 output features; this warp: 32 rows x QC = Fo/4 of them (16 or 32)
        const int QC = g.Fo >> 2;
        float4* pst = reinterpret_cast<float4*>(smem + PST_OFF + warp * (32 * QC * 4));
        const size_t row_base = ((size_t)dir * g.NSEQ + seq0 + q * 32) * T + tp;
        const int col0 = rank * (g.Fo >> 1) + e * QC;
        uint32_t a[32];
        if (QC == 32) ptx::tmem_ld32(tmem + lane_off + (uint32_t)(slot * 128 + e * QC), a);
        else ptx::tmem_ld16(tmem + lane_off + (uint32_t)(slot * 128 + e * QC), reinterpret_cast<uint32_t(&)[16]>(a));
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->accempty[slot]));
        if (QC == 32) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            pst[lane * 8 + (i ^ (lane & 7))] = make_float4(__uint_as_float(a[4 * i]) * sc.inv_p, __uint_as_float(a[4 * i + 1]) * sc.inv_p,
                                                           __uint_as_float(a[4 * i + 2]) * sc.inv_p, __uint_as_float(a[4 * i + 3]) * sc.inv_p);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int row = j * 4 + (lane >> 3), qq = lane & 7;
            const float4 v = pst[row * 8 + (qq ^ (row & 7))];
            if (seq0 + q * 32 + row < g.NSEQ) *reinterpret_cast<float4*>(g.P + (row_base + (size_t)row * T) * g.Fo + col0 + qq * 4) = v;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            pst[lane * 4 + (i ^ (lane & 3))] = make_float4(__uint_as_float(a[4 * i]) * sc.inv_p, __uint_as_float(a[4 * i + 1]) * sc.inv_p,
                                                           __uint_as_float(a[4 * i + 2]) * sc.inv_p, __uint_as_float(a[4 * i + 3]) * sc.inv_p);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int row = j * 8 + (lane >> 2), qq = lane & 3;
            const float4 v = pst[row * 4 + (qq ^ (row & 3))];
            if (seq0 + q * 32 + row < g.NSEQ) *reinterpret_cast<float4*>(g.P + (row_base + (size_t)row * T) * g.Fo + col0 + qq * 4) = v;
          }
        }
        __syncwarp();
        tl_mark(tl, t, 1, 4, 3);
        ++gidx;
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  ptx::cluster_sync_all();  // nobody leaves while the peer may still copy into / arrive on this CTA
  if (warp == 8) ptx::tmem_dealloc(tmem, 512);
}

// ---- operand preparation -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_absmax_flat(const float* __restrict__ x, size_t n, unsigned* __restrict__ out) {
  float m = 0.f;
  const size_t n4 = n / 4;
  const float4* p = reinterpret_cast<const float4*>(x);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(p + i);
    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  if (blockIdx.x == 0)
    for (size_t i = n4 * 4 + threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));  // non-negative floats order like their bit patterns
}

__device__ __forceinline__ float block_max(float m, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  float r = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r = fmaxf(r, red[i]);
  return r;
}
// smallest e with 2^e > m (m finite, > 0); clamped
__device__ __forceinline__ int ceil_exp(float m, int lo, int hi) {
  int e = m > 0.f ? (int)((__float_as_uint(m) >> 23) & 255u) - 126 : lo;
  return e < lo ? lo : (e > hi ? hi : e);
}
__device__ __forceinline__ float exp2i(int k) { return __uint_as_float((uint32_t)(k + 127) << 23); }

// max|W_ih|, max|W_hh|, max|W_fc[:, dir half]| per direction: grid (16, 2), atomicMax on the bit patterns into wmax[dir*3 + {0,1,2}]
__global__ void __launch_bounds__(256) k_lstm_wmax(const float* __restrict__ wih_f, const float* __restrict__ whh_f,
                                                   const float* __restrict__ wih_r, const float* __restrict__ whh_r,
                                                   const float* __restrict__ wfc, int F, int H, int Fo, unsigned* __restrict__ wmax) {
  __shared__ float red[32];
  const int d = blockIdx.y;
  const float* wih = d ? wih_r : wih_f;
  const float* whh = d ? whh_r : whh_f;
  float mi = 0.f, mh = 0.f, mp = 0.f;
  const int t0 = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  for (int i = t0; i < 4 * H * F; i += nt) mi = fmaxf(mi, fabsf(wih[i]));
  for (int i = t0; i < 4 * H * H; i += nt) mh = fmaxf(mh, fabsf(whh[i]));
  if (wfc)
    for (int i = t0; i < Fo * H; i += nt) mp = fmaxf(mp, fabsf(wfc[(size_t)(i / H) * 2 * H + d * H + (i % H)]));
  mi = block_max(mi, red);
  mh = block_max(mh, red);
  mp = block_max(mp, red);
  if (threadIdx.x == 0) {
    if (mi > 0.f) atomicMax(wmax + d * 3 + 0, __float_as_uint(mi));
    if (mh > 0.f) atomicMax(wmax + d * 3 + 1, __float_as_uint(mh));
    if (mp > 0.f) atomicMax(wmax + d * 3 + 2, __float_as_uint(mp));
  }
}

// power-of-two operand scales from max|x| (measured on this call's input) and this direction's max|W|
__device__ __forceinline__ LstmScales lstm_scales(const unsigned* __restrict__ xmax, const unsigned* __restrict__ wmax, int d) {
  const float mi = __uint_as_float(wmax[d * 3 + 0]), mh = __uint_as_float(wmax[d * 3 + 1]), mp = __uint_as_float(wmax[d * 3 + 2]);
  const int ex = ceil_exp(__uint_as_float(*xmax), -40, 40);
  const int eW = ceil_exp(fmaxf(mi * exp2i(ex), mh), -60, 60);
  const int eP = ceil_exp(mp, -60, 60);
  LstmScales s;
  s.x_mul = exp2i(14 - ex);
  s.w_ih_mul = exp2i(ex + 14 - eW);
  s.w_hh_mul = exp2i(14 - eW);
  s.inv_g = exp2i(eW - 28);
  s.w_p_mul = exp2i(14 - eP);
  s.inv_p = exp2i(eP - 28);
  s.pad[0] = s.pad[1] = 0.f;
  return s;
}

// grid (n_imgs, 2 directions, ranks): one 16 KB slab image per block.  Gate slab (chunk c, slab k): column n = 64 e + 4 u + gate <->
// weight row gate * H + 32 cg + 16 e + u (cg = global chunk), k-elements of [W_ih * w_ih_mul | W_hh * w_hh_mul]; projection slab k: row n =
// output feature, W_fc[n][dir * H + ...] * w_p_mul.  1-CTA kernel (ranks = 1): chunks 0..KSH-1, h slabs in natural order.  2-CTA
// kernel (ranks = 2): CTA `rank` gets chunks rank*CH + [0,CH), its h slabs ordered [own half | peer half], and rows
// rank*Fo/2 + [0,Fo/2) of the projection.  Block (0, dir, rank) also writes the bias table (pre-scaled ex2 arguments).
__global__ void __launch_bounds__(256) k_lstm_build(const float* __restrict__ wih_f, const float* __restrict__ whh_f,
                                                    const float* __restrict__ bih_f, const float* __restrict__ bhh_f,
                                                    const float* __restrict__ wih_r, const float* __restrict__ whh_r,
                                                    const float* __restrict__ bih_r, const float* __restrict__ bhh_r,
                                                    const float* __restrict__ wfc, int F, int H, int Fo, const unsigned* __restrict__ xmax,
                                                    const unsigned* __restrict__ wmax, LstmScales* __restrict__ scp,
                                                    uint8_t* __restrict__ img, float* __restrict__ bias, int n_imgs) {
  const int d = blockIdx.y, idx = blockIdx.x, rank = blockIdx.z, R = gridDim.z;
  const float* wih = d ? wih_r : wih_f;
  const float* whh = d ? whh_r : whh_f;
  const LstmScales sc = lstm_scales(xmax, wmax, d);
  if (idx == 0 && rank == 0 && threadIdx.x == 0) scp[d] = sc;  // the recurrence kernel reads them from here
  const int KSX = F / 32, KSH = H / 32, CH = KSH / R, per = KSX + KSH, n_gate = CH * per;
  uint8_t* dst = img + ((size_t)(d * R + rank) * n_imgs + idx) * SLAB_BYTES;
  auto hslab = [&](int kh) { return R == 1 ? kh : (kh < CH ? rank * CH + kh : (1 - rank) * CH + (kh - CH)); };
  if (idx == 0) {
    const float* bi = d ? bih_r : bih_f;
    const float* bh = d ? bhh_r : bhh_f;
    for (int i = threadIdx.x; i < 128 * CH; i += blockDim.x) {
      const int c = i / 128, n = i % 128, row = (n & 3) * H + 32 * (rank * CH + c) + 16 * (n >> 6) + ((n & 63) >> 2);
      // stored as the ex2 argument's additive term: -log2(e) b for i, f, o; -2 log2(e) b for g (gate index 2)
      bias[(size_t)(d * R + rank) * 128 * CH + i] = (bi[row] + bh[row]) * ((n & 3) == 2 ? -2.8853900817779268f : -1.4426950408889634f);
    }
  }
  const bool is_proj = idx >= n_gate;
  const int rows = is_proj ? Fo / R : 128;
  const uint32_t lo_base = (uint32_t)rows * 64u;
  const int c = is_proj ? 0 : idx / per, k = is_proj ? idx - n_gate : idx % per;
  for (int i = threadIdx.x; i < rows * 16; i += blockDim.x) {  // one pair of k-elements per iteration
    const int n = i / 16, kk = (i % 16) * 2;
    float v0, v1;
    if (is_proj) {
      const float* p = wfc + (size_t)(rank * (Fo / R) + n) * 2 * H + d * H + 32 * hslab(k) + kk;
      v0 = p[0] * sc.w_p_mul;
      v1 = p[1] * sc.w_p_mul;
    } else {
      const int row = (n & 3) * H + 32 * (rank * CH + c) + 16 * (n >> 6) + ((n & 63) >> 2);
      if (k < KSX) {
        const float* p = wih + (size_t)row * F + 32 * k + kk;
        v0 = p[0] * sc.w_ih_mul;
        v1 = p[1] * sc.w_ih_mul;
      } else {
        const float* p = whh + (size_t)row * H + 32 * hslab(k - KSX) + kk;
        v0 = p[0] * sc.w_hh_mul;
        v1 = p[1] * sc.w_hh_mul;
      }
    }
    uint32_t hi, lo;
    ptx::split_f16x2(v0, v1, hi, lo);
    const uint32_t off = (uint32_t)(n >> 3) * 512u + (uint32_t)(n & 7) * 64u + ((((uint32_t)kk >> 3) ^ (((uint32_t)n >> 1) & 3u)) << 4) +
                         ((uint32_t)kk & 7u) * 2u;
    *reinterpret_cast<uint32_t*>(dst + off) = hi;
    *reinterpret_cast<uint32_t*>(dst + lo_base + off) = lo;
  }
}

// Y = P0 + P1 + bias (the Linear of dprnn.py:87 / 139 split over the two directions): gLN statistics of it ...
__global__ void __launch_bounds__(256) k_sample_stats2(const float* __restrict__ P0, const float* __restrict__ P1,
                                                       const float* __restrict__ bias, size_t n, int F, double* __restrict__ stats) {
  __shared__ double red[64];
  const int b = blockIdx.y;
  const float4* p0 = reinterpret_cast<const float4*>(P0 + (size_t)b * n);
  const float4* p1 = reinterpret_cast<const float4*>(P1 + (size_t)b * n);
  const size_t n4 = n / 4;  // F % 4 == 0
  double s = 0.0, ss = 0.0;
  for (size_t i0 = (size_t)blockIdx.x * blockDim.x * 4; i0 < n4; i0 += (size_t)gridDim.x * blockDim.x * 4) {
    float ls = 0.f, lss = 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const size_t i = i0 + (size_t)u * blockDim.x + threadIdx.x;
      if (i < n4) {
        const float4 a = __ldg(p0 + i), c = __ldg(p1 + i), bb = __ldg(reinterpret_cast<const float4*>(bias + (i * 4) % F));
        const float x = a.x + c.x + bb.x, y = a.y + c.y + bb.y, z = a.z + c.z + bb.z, w = a.w + c.w + bb.w;
        ls += (x + y) + (z + w);
        lss = fmaf(x, x, fmaf(y, y, fmaf(z, z, fmaf(w, w, lss))));
      }
    }
    s += ls;
    ss += lss;
  }
  block_sum2_d(s, ss, red);
  if (threadIdx.x == 0) { atomicAdd(&stats[2 * b], s); atomicAdd(&stats[2 * b + 1], ss); }
}

// ... and out = gLN(Y) + R, optionally stored with the two middle dimensions swapped (the layout of the other path).
// grid (D1, B), block (F/4, 256/(F/4)): one block per (b, d1) row of D2 x F floats (contiguous on the read side: a warp reads 512
// consecutive bytes of each operand); 4 independent cells per thread in flight; on the swapped side every cell is one 4F-byte run.
__global__ void __launch_bounds__(256) k_norm_res2(const float* __restrict__ P0, const float* __restrict__ P1, const float* __restrict__ bias,
                                                   const float* __restrict__ R, const float* __restrict__ gamma,
                                                   const float* __restrict__ beta, float* __restrict__ out, const double* __restrict__ stats,
                                                   int D1, int D2, int F, float eps, int swap, unsigned* __restrict__ absmax) {
  const int b = blockIdx.y, d1 = blockIdx.x, f = threadIdx.x * 4;
  float amax = 0.f;
  const float2 mr = gln_mean_rstd(stats + 2 * b, (double)D1 * (double)D2 * (double)F, eps);
  const float4 bb = __ldg(reinterpret_cast<const float4*>(bias + f)), gm = __ldg(reinterpret_cast<const float4*>(gamma + f)),
               be = __ldg(reinterpret_cast<const float4*>(beta + f));
  // y_norm = (p0 + p1 + bias - mean) * rstd * gamma + beta  ==  (p0 + p1) * sc + sh
  const float4 sc = make_float4(mr.y * gm.x, mr.y * gm.y, mr.y * gm.z, mr.y * gm.w);
  const float4 sh = make_float4(fmaf(bb.x - mr.x, sc.x, be.x), fmaf(bb.y - mr.x, sc.y, be.y), fmaf(bb.z - mr.x, sc.z, be.z),
                                fmaf(bb.w - mr.x, sc.w, be.w));
  const size_t row = ((size_t)b * D1 + d1) * D2;
  const int TY = blockDim.y;
  for (int d20 = threadIdx.y; d20 < D2; d20 += 4 * TY) {
    float4 a[4], c[4], r[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int d2 = d20 + u * TY;
      if (d2 < D2) {
        const size_t src = (row + d2) * F + f;
        a[u] = __ldg(reinterpret_cast<const float4*>(P0 + src));
        c[u] = __ldg(reinterpret_cast<const float4*>(P1 + src));
        r[u] = __ldg(reinterpret_cast<const float4*>(R + src));
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int d2 = d20 + u * TY;
      if (d2 < D2) {
        const size_t dst = (swap ? ((size_t)b * D2 + d2) * D1 + d1 : row + d2) * F + f;
        float4 o;
        o.x = fmaf(a[u].x + c[u].x, sc.x, sh.x) + r[u].x;
        o.y = fmaf(a[u].y + c[u].y, sc.y, sh.y) + r[u].y;
        o.z = fmaf(a[u].z + c[u].z, sc.z, sh.z) + r[u].z;
        o.w = fmaf(a[u].w + c[u].w, sc.w, sh.w) + r[u].w;
        *reinterpret_cast<float4*>(out + dst) = o;
        amax = fmaxf(amax, fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))));
      }
    }
  }
  if (absmax) {  // max|out|: the operand scale of the next path's LSTM (saves its own pass over the state)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if (((threadIdx.y * blockDim.x + threadIdx.x) & 31) == 0 && amax > 0.f) atomicMax(absmax, __float_as_uint(amax));
  }
}

struct LstmPlan {
  int n_imgs, n_st, pair;
  size_t off_sc, off_bias, off_img, total, smem;
};
bool lstm_plan(int F, int H, int Fo, LstmPlan& p, bool allow_pair = true) {
  if (!(H == 32 || H == 64 || H == 128) || !(F == 32 || F == 64 || F == 128)) return false;
  if (Fo != 0 && (Fo % 32 != 0 || Fo < 32 || Fo > 128)) return false;
  const int KSX = F / 32, KSH = H / 32;
  // 2-CTA form: H >= 64 (each CTA needs whole 32-unit chunks) and Fo/4 a multiple of 16 (store granularity of a warp)
  p.pair = (allow_pair && KSH >= 2 && (Fo == 0 || Fo == 64 || Fo == 128)) ? 1 : 0;
  if (const char* e = getenv("CTN_LSTM_PAIR")) p.pair = p.pair && atoi(e) != 0;
  const int R = p.pair ? 2 : 1, CH = KSH / R;
  p.n_imgs = CH * (KSX + KSH) + KSH;
  p.off_sc = 256;
  p.off_bias = 512;
  p.off_img = 512 + (((size_t)2 * 4 * H * sizeof(float) + 255) / 256) * 256;
  p.total = p.off_img + (size_t)2 * R * p.n_imgs * SLAB_BYTES;
  size_t fixed;
  int n_st;
  if (p.pair) {
    fixed = 1024 /*alignment slack*/ + 2 * HDR_BYTES + (size_t)256 * (Fo ? Fo : 64) + (size_t)4 * CH * SLAB_BYTES;
    n_st = (int)((232448 - fixed) / SLAB_BYTES);
    if (n_st > PAIR_MAX_ST) n_st = PAIR_MAX_ST;
  } else {
    fixed = 1024 + HDR_BYTES + 2048 + (size_t)2 * KSX * 8192 + PSTAGE_BYTES;
    n_st = (int)((232448 - fixed) / STAGE_BYTES);
    if (n_st > MAX_ST) n_st = MAX_ST;
  }
  if (const char* e = getenv("CTN_LSTM_STAGES")) { const int v = atoi(e); if (v >= 2 && v < n_st) n_st = v; }
  if (n_st < 2) return false;
  p.n_st = n_st;
  p.smem = fixed + (size_t)n_st * (p.pair ? SLAB_BYTES : STAGE_BYTES);
  return true;
}

template <int NCH, int KSX>
int launch_bilstm(const LstmArgs& a, size_t smem, cudaStream_t st) {
  static bool done[CTN_MAX_DEVICES] = {};
  const int dev = ctn_current_device();
  if (!done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_bilstm<NCH, KSX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return (int)e;
    done[dev] = true;
  }
  k_bilstm<NCH, KSX><<<dim3((a.NSEQ + LM - 1) / LM, 2), LSTM_THREADS, smem, st>>>(a);
  return CTN_OK;
}

template <int NCH, int KSX>
int launch_bilstm_pair(const LstmArgs& a, size_t smem, cudaStream_t st) {
  static bool done[CTN_MAX_DEVICES] = {};
  const int dev = ctn_current_device();
  if (!done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_bilstm_pair<NCH, KSX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return (int)e;
    done[dev] = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * ((a.NSEQ + LM - 1) / LM), 2);
  cfg.blockDim = dim3(LSTM_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, k_bilstm_pair<NCH, KSX>, a);
  return e == cudaSuccess ? CTN_OK : (int)e;
}

}  // namespace

// debug: copies the timeline probe (see g_lstm_tl) to the host; n <= 160
extern "C" int ctn_debug_lstm_timeline(unsigned long long* out, int n) {
  if (!out || n <= 0 || n > 160) return CTN_EINVAL;
  cudaError_t e = cudaMemcpyFromSymbol(out, g_lstm_tl, sizeof(unsigned long long) * n);
  return e == cudaSuccess ? CTN_OK : (int)e;
}

extern "C" int ctn_bilstm_supported(int F, int H, int Fo) {
  LstmPlan p;
  return lstm_plan(F, H, Fo, p) ? 1 : 0;
}

extern "C" size_t ctn_bilstm_workspace_bytes(int F, int H, int Fo) {
  LstmPlan p;
  return lstm_plan(F, H, Fo, p) ? p.total : 0;
}

extern "C" int ctn_bilstm_proj_fwd(const float* z, int NSEQ, int T, int F, int H, const float* const* w, const float* w_fc, int Fo, float* P,
                                   float* hout, const unsigned* z_absmax, void* workspace, size_t workspace_bytes, ctn_stream_t stream) {
  LaunchScope scope(z);
  if (!z || !w || !workspace || NSEQ <= 0 || T <= 0) return CTN_EINVAL;
  for (int i = 0; i < 8; ++i)
    if (!w[i]) return CTN_EINVAL;
  if ((w_fc == nullptr) != (P == nullptr)) return CTN_EINVAL;
  if (!w_fc && !hout) return CTN_EINVAL;
  LstmPlan p;
  if (!lstm_plan(F, H, w_fc ? Fo : 0, p)) return CTN_EUNSUPPORTED;
  if (workspace_bytes < p.total) return CTN_EWORKSPACE;
  if (p.pair && !getenv("CTN_LSTM_PAIR")) {
    // the 2-CTA form halves the time of a step but needs twice the CTAs: worth it only while they all fit on the GPU at once
    if (4 * ((NSEQ + LM - 1) / LM) > ctn_num_sms() && !lstm_plan(F, H, w_fc ? Fo : 0, p, false)) return CTN_EUNSUPPORTED;
  }
  if ((((uintptr_t)z) | ((uintptr_t)P) | ((uintptr_t)hout) | ((uintptr_t)workspace)) & 15) return CTN_EALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  unsigned* xmax = reinterpret_cast<unsigned*>(ws);
  LstmScales* sc = reinterpret_cast<LstmScales*>(ws + p.off_sc);
  float* bias = reinterpret_cast<float*>(ws + p.off_bias);
  uint8_t* img = ws + p.off_img;
  unsigned* wmax = xmax + 1;  // [2][3]
  cudaError_t e = cudaMemsetAsync(xmax, 0, 32, st);
  if (e != cudaSuccess) return (int)e;
  const size_t n = (size_t)NSEQ * T * F;
  int gx = (int)((n / 4 + 255) / 256);
  if (gx > 1184) gx = 1184;
  if (gx < 1) gx = 1;
  if (z_absmax) {
    xmax = const_cast<unsigned*>(z_absmax);  // supplied by the producer of z (ctn_dprnn_norm_res2_fwd): bit pattern of max|z|
  } else {
    k_absmax_flat<<<gx, 256, 0, st>>>(z, n, xmax);
    CTN_COUNT_LAUNCH();
  }
  // w: weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0, then the same four with the _reverse suffix (torch.nn.LSTM names)
  k_lstm_wmax<<<dim3(16, 2), 256, 0, st>>>(w[0], w[1], w[4], w[5], w_fc, F, H, Fo, wmax);
  CTN_COUNT_LAUNCH();
  const int n_build = w_fc ? p.n_imgs : p.n_imgs - H / 32;
  k_lstm_build<<<dim3(n_build, 2, p.pair ? 2 : 1), 256, 0, st>>>(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], w_fc, F, H, Fo, xmax, wmax, sc, img, bias, p.n_imgs);
  CTN_COUNT_LAUNCH();
  LstmArgs a;
  a.z = z; a.P = P; a.hout = hout; a.img = img; a.bias = bias; a.sc = sc;
  a.NSEQ = NSEQ; a.T = T; a.Fo = w_fc ? Fo : 32; a.n_imgs = p.n_imgs; a.n_st = p.n_st; a.has_proj = w_fc ? 1 : 0;
  a.dbg = 0;
  if (const char* e = getenv("CTN_LSTM_DBG")) a.dbg = (uint32_t)atoi(e);
  int rc = CTN_EUNSUPPORTED;
  const int NCH = H / 32, KSX = F / 32;
#define CTN_LSTM_CASE(nch, ksx) if (NCH == nch && KSX == ksx) rc = launch_bilstm<nch, ksx>(a, p.smem, st);
#define CTN_LSTM_PAIR_CASE(nch, ksx) if (NCH == nch && KSX == ksx) rc = launch_bilstm_pair<nch, ksx>(a, p.smem, st);
  if (p.pair) {
    CTN_LSTM_PAIR_CASE(2, 1) CTN_LSTM_PAIR_CASE(2, 2) CTN_LSTM_PAIR_CASE(2, 4) CTN_LSTM_PAIR_CASE(4, 1) CTN_LSTM_PAIR_CASE(4, 2)
    CTN_LSTM_PAIR_CASE(4, 4)
  } else {
    CTN_LSTM_CASE(1, 1) CTN_LSTM_CASE(2, 1) CTN_LSTM_CASE(2, 2) CTN_LSTM_CASE(4, 1) CTN_LSTM_CASE(4, 2) CTN_LSTM_CASE(4, 4)
    CTN_LSTM_CASE(1, 2) CTN_LSTM_CASE(1, 4) CTN_LSTM_CASE(2, 4)
  }
#undef CTN_LSTM_CASE
#undef CTN_LSTM_PAIR_CASE
  if (rc != CTN_OK) return rc;
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

extern "C" int ctn_dprnn_norm_res2_fwd(const float* P, const float* fc_bias, const float* R, const float* gamma, const float* beta,
                                       float* out, int B, int D1, int D2, int F, float eps, int swap, double* scratch, unsigned* out_absmax,
                                       ctn_stream_t stream) {
  LaunchScope scope(P);
  if (!P || !fc_bias || !R || !gamma || !beta || !out || !scratch || B <= 0 || D1 <= 0 || D2 <= 0 || F <= 0 || (F & 3)) return CTN_EINVAL;
  if (F > 1024 || D1 > 65535 * 32 || B > 65535) return CTN_EUNSUPPORTED;
  if (swap && out == R) return CTN_EINVAL;
  if ((((uintptr_t)P) | ((uintptr_t)R) | ((uintptr_t)out) | ((uintptr_t)gamma) | ((uintptr_t)beta) | ((uintptr_t)fc_bias)) & 15)
    return CTN_EALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(scratch, 0, sizeof(double) * 2 * B, st);
  if (e != cudaSuccess) return (int)e;
  if (out_absmax && (e = cudaMemsetAsync(out_absmax, 0, sizeof(unsigned), st)) != cudaSuccess) return (int)e;
  const size_t n = (size_t)D1 * D2 * F;
  const float* P1 = P + (size_t)B * n;  // second direction
  int gx = (int)((n / 4 + 256 * 4 - 1) / (256 * 4));
  {  // ~8 resident blocks per SM over the WHOLE batch: longer per-thread streams, 2 double atomics per block on 2B addresses
    const int cap = 1184 / B > 1 ? 1184 / B : 1;
    if (gx > cap) gx = cap;
  }
  if (gx < 1) gx = 1;
  k_sample_stats2<<<dim3(gx, B), 256, 0, st>>>(P, P1, fc_bias, n, F, scratch);
  CTN_COUNT_LAUNCH();
  const int q = F / 4;
  k_norm_res2<<<dim3(D1, B), dim3(q, 256 / q >= 1 ? 256 / q : 1), 0, st>>>(P, P1, fc_bias, R, gamma, beta, out, scratch, D1, D2, F, eps, swap, out_absmax);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}
