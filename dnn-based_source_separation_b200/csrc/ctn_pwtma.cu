// TMA-fed tcgen05 kernels for the two dense contractions of a TCN block (src/models/tdcn.py:107-196), fp16-piece mode.
//
//   pw1:  h = PReLU(W1 x + b1) (+ gLN1 statistics);  x = x_prev + deferred gLN2 update of the previous block   (PRO_RES / PRO_NONE, EPI_H)
//   pw2:  r = [Wo;Ws] diag(gamma2) u,  u = PReLU(dwconv_d(zero-pad(gLN1(h))) + bd) formed on the fly            (PRO_DW, EPI_RAW)
//
// Same orientation, operand layouts, weight images, TMEM accumulator ring and epilogues as k_pw_umma (ctn_umma.cu).  What
// changes is how the activation operand reaches the producers: in k_pw_umma every producer thread issues its own LDG.128s
// and then waits a full L2/HBM latency per slab (ncu: 60-70 % of the producers' stall samples are long-scoreboard waits
// right behind the loads; only ONE slab of loads is in flight per thread).  Here ONE elected thread issues tensor-map TMA
// box loads (cp.async.bulk.tensor.2d, mbarrier complete_tx) of RAW fp32 tiles into a shared-memory ring that runs several
// 16-channel stages ahead; the producer warps read the raw tiles with LDS (~30 cycles), apply the prologue, split into fp16
// hi/lo pieces and store the swizzled MN-major operand.  The global-load latency is hidden by the depth of the raw ring
// instead of by registers, the dilated halo of the depthwise conv is ONE box of 128 + 2d frames (d <= 64) or three boxes
// (d >= 128) instead of 3 loads per thread, and the per-channel parameters travel with the tile (one 512-byte bulk copy).
//
// fp16 envelope: every activation operand is multiplied by a power of two `act_scale` chosen per forward from a bound
// derived from the weights alone (ctn_act_scales, ctn_tcn_simt.cu), so that |operand| <= 2^15 ALWAYS holds (no saturation,
// whatever the checkpoint) -- the epilogue multiplies the exact inverse back together with the weight-group scales.
//
// Warp roles (one persistent CTA per SM):
//   0-3    epilogue group 0            4  TMEM allocator + MMA issuer        5  TMA loader (one elected lane)
//   6..13  producers: 8 warps, each 2 channels of each of the two 16-channel raw stages of a slab (4 interleaved channel streams)
//   then   epilogue group 1 (EPI_H kernels: 4 more warps, upper half of the columns)
#include <cuda.h>
#include <cuda_fp16.h>
#include <string.h>
#include "ctn_internal.h"
#include "ctn_umma_ptx.cuh"
#include "ctn_dw_math.cuh"

namespace {

constexpr int TM = 128;      // time steps per tile (UMMA M)
constexpr int KS = 32;       // input channels per operand slab
constexpr int RC = 16;       // channels per raw (TMA) stage
constexpr int SUBS = KS / RC;
constexpr int A_BYTES = TM * KS * 2;  // one fp16 precision of an activation slab
constexpr int MAX_OP = 6, MAX_RAW = 8;
constexpr int HDR_FIXED = 2048;       // barriers + tmem pointer, then float[256] epilogue parameters at +1024
constexpr int SMEM_PARAMS = 1024;

struct TmaArgs {
  PwArgs a;
  CUtensorMap tmA;  // activation operand, 2-D (pitch, B*K) fp32
  CUtensorMap tmR;  // PRO_RES: raw [out;skip] contraction of the previous block, 2-D (pitch, B*res_Mt)
  const uint8_t* wimg;
  const float* oscale;
  const float* dwp;        // PRO_DW: packed per-channel parameters [ceil16(K)][8] = {gamma1, beta1, w0, w1, w2, bd, 0, 0}
  const float* act_scale;  // power-of-two scale of the activation operand (device scalar; nullable = 1)
  int n_tile, n_tiles, k_slabs, t_tiles, num_items;
  int op_stages, raw_stages;
  uint32_t op_stage_bytes, raw_stage_bytes, raw_tx_bytes, w_bytes, hdr_bytes, res_tab_off, idesc;
  int reverse;   // walk the (sample, time tile) list backwards
  int dw_three;  // PRO_DW: 0 = one window box of 128 + 2*dw_pad frames, 1 = three boxes of 128 frames at t-d, t, t+d
  int dw_pad;    // window mode: halo frames on each side (dilation rounded up to a multiple of 4)
};

template <int PRO> struct Roles {
  // x SUBS * CPW channel streams per warp and slab.  The mask kernel's prologue (PReLU of the skip sum, K = 128) is light: 4 producer
  // warps keep the CTA at 448 threads, i.e. 144 instead of 96 registers per thread for its heavy epilogue (sigmoid, w * mask, decoder taps)
  static constexpr int PROD_WARPS = PRO == PRO_PRELU ? 4 : 8;
  static constexpr int EGROUPS = PRO == PRO_DW ? 1 : 2;
  static constexpr int FIRST_PROD = 6;
  static constexpr int THREADS = (4 + 1 + 1 + PROD_WARPS + 4 * (EGROUPS - 1)) * 32;
};

struct __align__(8) Header {
  uint64_t full[MAX_OP], empty[MAX_OP];      // operand ring (A pieces + W slab)
  uint64_t rfull[MAX_RAW], rempty[MAX_RAW];  // raw ring
  uint64_t tfull[2], tempty[2];              // TMEM accumulator ring
  uint32_t tmem_base;
};
static_assert(sizeof(Header) <= SMEM_PARAMS, "header");

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(bar)
               : "memory");
}
// arrive on a "slot free" barrier AFTER the values read from the slot exist in registers: `dep` (a value computed from them) is an
// input operand, so the arrive cannot issue while the shared-memory loads are still in flight (a release does not wait for
// outstanding LDS by itself; the TMA engine would otherwise overwrite the slot under them)
__device__ __forceinline__ void mbar_arrive_after(uint32_t bar, float dep) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar), "f"(dep) : "memory");
}
// shared-memory accesses of the producers' inner loop by 32-bit shared address (a generic pointer costs an S2R/LEA/IADD
// window-base computation per access: 15 % of the producers' instructions in the ncu source view)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t lo, uint32_t hi) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(lo), "r"(hi) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

// DWM (PRO_DW only): depthwise tap geometry fixed at compile time -- 1 / 2: dilation 1 / 2 in the aligned window [t-4, t+8);
// 3: dilation >= 4, one window box of 128 + 2d frames; 4: dilation >= 128, three boxes of 128 frames.  0 for the other prologues.
template <int PRO, int EPI, int DWM>
__global__ void __launch_bounds__(Roles<PRO>::THREADS, 1) k_pw_tma(const __grid_constant__ TmaArgs g) {
  constexpr bool TRAIN = (DWM & 8) != 0;  // training forward: PReLU on load, u_pre stored (see PwArgs::dw_in_slope)
  constexpr int DCLS = (DWM & 7) == 1 ? 1 : ((DWM & 7) == 2 ? 2 : 4);
  constexpr bool THREE = (DWM & 7) == 4;
  constexpr int PROD_WARPS = Roles<PRO>::PROD_WARPS, EGROUPS = Roles<PRO>::EGROUPS, FIRST_PROD = Roles<PRO>::FIRST_PROD;
  constexpr int CPW = RC / PROD_WARPS;  // channels of a raw stage per producer warp (1 or 2)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  Header* hdr = reinterpret_cast<Header*>(smem);
  float* ssc_all = reinterpret_cast<float*>(smem + HDR_FIXED);  // per padded output channel: weight-group scale / act_scale
  const uint32_t op0 = base + g.hdr_bytes;
  const uint32_t raw0 = op0 + (uint32_t)g.op_stages * g.op_stage_bytes;
  uint8_t* const raw0_p = smem + g.hdr_bytes + (size_t)g.op_stages * g.op_stage_bytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const PwArgs& a = g.a;

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.op_stages; ++s) {
      ptx::mbar_init(ptx::smem_u32(&hdr->full[s]), PROD_WARPS + 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->empty[s]), 1);
    }
    for (int s = 0; s < g.raw_stages; ++s) {
      ptx::mbar_init(ptx::smem_u32(&hdr->rfull[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->rempty[s]), PROD_WARPS);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(ptx::smem_u32(&hdr->tfull[i]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->tempty[i]), 128 * EGROUPS);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 4) ptx::tmem_alloc(ptx::smem_u32(&hdr->tmem_base), 512);
  if (warp == 5 && lane == 0) {
    tma_prefetch_desc(&g.tmA);
    if (PRO == PRO_RES) tma_prefetch_desc(&g.tmR);
  }
  const float act_s = g.act_scale ? __ldg(g.act_scale) : 1.f;
  {
    const float inv = 1.f / act_s;  // power of two: exact
    for (int i = threadIdx.x; i < g.n_tiles * g.n_tile; i += blockDim.x) ssc_all[i] = __ldg(g.oscale + i) * inv;
  }
  float* s_res = reinterpret_cast<float*>(smem + g.res_tab_off);  // [2][k_slabs*KS]: v1, v2 (zero past K)
  if (PRO == PRO_RES) {
    const int kp = g.k_slabs * KS;
    for (int i = threadIdx.x; i < kp; i += blockDim.x) {
      s_res[i] = i < a.K ? __ldg(a.res_v1 + i) : 0.f;
      s_res[kp + i] = i < a.K ? __ldg(a.res_v2 + i) : 0.f;
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = hdr->tmem_base;

  // EPI_MASKDEC: a CTA walks ALL n-tiles of a (sample, time tile) back to back (the decoder sums over the channels of a source
  // in registers); the other kernels interleave n-tiles across CTAs (n-tile fastest, co-running CTAs share activations in L2)
  const int tiles_total = g.num_items / g.n_tiles;
  const int cta = (int)blockIdx.x, ncta = (int)gridDim.x;
  const int items_per_cta = EPI == EPI_MASKDEC ? ((tiles_total - cta + ncta - 1) / ncta) * g.n_tiles
                                               : (g.num_items - cta + ncta - 1) / ncta;
  auto decode = [&](int it2, int& nt2, int& tt2, int& b2) {
    int L;
    if (EPI == EPI_MASKDEC) {
      nt2 = it2 % g.n_tiles;
      L = cta + (it2 / g.n_tiles) * ncta;
    } else {
      const int J = cta + it2 * ncta;
      nt2 = J % g.n_tiles;
      L = J / g.n_tiles;
    }
    // reverse walk (pw2): the previous kernel (pw1, forward) wrote the LAST samples' h most recently -- start with what is still in L2
    if (g.reverse) L = tiles_total - 1 - L;
    tt2 = L % g.t_tiles;
    b2 = L / g.t_tiles;
  };
  if (EPI == EPI_MASKDEC) {
    // decoder basis (Nb x 16 taps) resident in shared memory behind the raw ring, then the [2][128][16] combine buffer
    float* sD = reinterpret_cast<float*>(raw0_p + (size_t)g.raw_stages * g.raw_stage_bytes);
    for (int i = threadIdx.x; i < a.Nb * 16; i += blockDim.x) sD[i] = __ldg(a.dec_w + i);
    __syncthreads();
  }

  if (warp == 5) {
    // ===================================== TMA LOADER ========================================================
    if (ptx::elect_one()) {
      int s = 0, rs = 0;
      uint32_t ph = 0, rph = 0;
      for (int it = 0; it < items_per_cta; ++it) {
        int nt, tt, b;
        decode(it, nt, tt, b);
        const uint8_t* wsrc = g.wimg + (size_t)nt * g.k_slabs * 2 * g.w_bytes;
        for (int ks = 0; ks < g.k_slabs; ++ks) {
#pragma unroll
          for (int sub = 0; sub < SUBS; ++sub) {
            ptx::mbar_wait(ptx::smem_u32(&hdr->rempty[rs]), rph ^ 1u);
            const uint32_t fb = ptx::smem_u32(&hdr->rfull[rs]);
            const uint32_t dst = raw0 + (uint32_t)rs * g.raw_stage_bytes;
            const int c = ks * KS + sub * RC;  // first channel of the stage
            ptx::mbar_arrive_expect_tx(fb, g.raw_tx_bytes);
            if (PRO == PRO_DW) {
              if (THREE) {
#pragma unroll
                for (int k = 0; k < 3; ++k)
                  tma_load_2d(dst + (uint32_t)k * (RC * TM * 4), &g.tmA, tt * TM + (k - 1) * a.dw_dilation, b * a.K + c, fb);
                ptx::bulk_g2s(dst + 3u * (RC * TM * 4), g.dwp + (size_t)c * 8, RC * 32, fb);
              } else {
                tma_load_2d(dst, &g.tmA, tt * TM - g.dw_pad, b * a.K + c, fb);
                ptx::bulk_g2s(dst + (uint32_t)(RC * (TM + 2 * g.dw_pad) * 4), g.dwp + (size_t)c * 8, RC * 32, fb);
              }
            } else {
              tma_load_2d(dst, &g.tmA, tt * TM, b * a.K + c, fb);
              if (PRO == PRO_RES) tma_load_2d(dst + RC * TM * 4, &g.tmR, tt * TM, b * a.res_Mt + c, fb);
            }
            if (++rs == g.raw_stages) { rs = 0; rph ^= 1u; }
          }
          ptx::mbar_wait(ptx::smem_u32(&hdr->empty[s]), ph ^ 1u);
          const uint32_t fb = ptx::smem_u32(&hdr->full[s]);
          ptx::mbar_arrive_expect_tx(fb, 2 * g.w_bytes);
          ptx::bulk_g2s(op0 + (uint32_t)s * g.op_stage_bytes + 2 * A_BYTES, wsrc + (size_t)ks * 2 * g.w_bytes, 2 * g.w_bytes, fb);
          if (++s == g.op_stages) { s = 0; ph ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= FIRST_PROD && warp < FIRST_PROD + PROD_WARPS) {
    // ===================================== PRODUCERS ========================================================
    // One step = one 32-channel operand slab = TWO raw stages; every warp works on SUBS * CPW = 4 independent channel streams
    // per step (knob matrix of round 2: the producers alone took 104 us per pw2 launch at ~10 cycles per instruction and warp --
    // dependent LDS -> FMA -> cvt -> STS chains, not issue slots; four interleaved streams per warp give the scheduler the
    // instruction-level parallelism, and the fence / full-arrive / empty-wait are paid once per slab instead of per 16 channels)
    const int pw = warp - FIRST_PROD;
    float pslope = 0.f, in_slope = 1.f;
    if (PRO == PRO_PRELU || PRO == PRO_DW) pslope = a.pro_slope[0];
    if (TRAIN) in_slope = a.dw_in_slope[0];
    int s = 0, rs = 0;
    uint32_t ph = 0, rph = 0;
    const int dw_wd = TM + 2 * g.dw_pad;  // PRO_DW window mode: floats per channel row of a raw stage
    for (int it = 0; it < items_per_cta; ++it) {
      int nt, tt, b;
      decode(it, nt, tt, b);
      float2 mr1 = make_float2(0.f, 1.f), mr_res = make_float2(0.f, 1.f);
      float2 dls = make_float2(0.f, 0.f), dlss = make_float2(0.f, 0.f);
      if (PRO == PRO_DW) mr1 = gln_mean_rstd(a.dw_stats_in + 2 * b, (double)a.K * (double)a.frames, a.dw_eps);
      if (PRO == PRO_RES) mr_res = gln_mean_rstd(a.res_stats + 2 * b, a.res_n, a.res_eps);
      const int tbase = tt * TM + lane * 4;
      bool dw_interior = false;
      if (PRO == PRO_DW) {
        const int d = a.dw_dilation;
        const int reach = DCLS == 4 ? d : 4;
        dw_interior = (tt * TM - reach >= 0) && (tt * TM + TM - 1 + reach + 3 < a.frames) && (a.K % RC == 0);
      }
      for (int ks = 0; ks < g.k_slabs; ++ks) {
        // the two raw stages of this slab (the ring may wrap between them)
        int rsv[SUBS];
        uint32_t rphv[SUBS];
#pragma unroll
        for (int sub = 0; sub < SUBS; ++sub) {
          rsv[sub] = rs; rphv[sub] = rph;
          if (++rs == g.raw_stages) { rs = 0; rph ^= 1u; }
        }
        float4 v[SUBS][CPW];
        float dep = 0.f;
#pragma unroll
        for (int sub = 0; sub < SUBS; ++sub) {
          ptx::mbar_wait(ptx::smem_u32(&hdr->rfull[rsv[sub]]), rphv[sub]);
          const uint32_t rb_s = raw0 + (uint32_t)rsv[sub] * g.raw_stage_bytes;  // shared address of the raw stage
          if (PRO == PRO_DW) {
            // u[c][t] = PReLU( sum_k wd[c][k] * hn[c][t + (k-1)*d] + bd[c] ), hn = gLN1(h) inside [0,frames), 0 outside
            const int d = a.dw_dilation;
            // tap loads: window mode -- the thread's first tap sits lane*4 floats into its channel row (the window starts `pad`
            // frames before the tile and pad == max(d, 4)); three-box mode -- same column in the boxes at t-d, t, t+d
            const uint32_t step_b = 4u * (uint32_t)(THREE ? RC * TM : (DCLS == 4 ? d : 4));
            const int tstep = DCLS == 4 ? d : 4;
            const int first = DCLS == 4 ? tbase - d : tbase - 4;
#pragma unroll
            for (int j = 0; j < CPW; ++j) {
              const int cl = pw * CPW + j;  // channel within the raw stage
              const int c = ks * KS + sub * RC + cl;
              const uint32_t qa = rb_s + 4u * (uint32_t)((THREE ? cl * TM : cl * dw_wd) + lane * 4);
              const uint32_t pa = rb_s + 4u * (uint32_t)((THREE ? 3 * RC * TM : RC * dw_wd) + cl * 8);
              float4 q0 = lds128(qa), q1 = lds128(qa + step_b), q2 = lds128(qa + 2 * step_b);
              const float4 p0 = lds128(pa), p1 = lds128(pa + 16);
              if (TRAIN) {  // the stored tensor is the pre-activation W1 x + b1
                q0.x = prelu_f(q0.x, in_slope); q0.y = prelu_f(q0.y, in_slope); q0.z = prelu_f(q0.z, in_slope); q0.w = prelu_f(q0.w, in_slope);
                q1.x = prelu_f(q1.x, in_slope); q1.y = prelu_f(q1.y, in_slope); q1.z = prelu_f(q1.z, in_slope); q1.w = prelu_f(q1.w, in_slope);
                q2.x = prelu_f(q2.x, in_slope); q2.y = prelu_f(q2.y, in_slope); q2.z = prelu_f(q2.z, in_slope); q2.w = prelu_f(q2.w, in_slope);
              }
              // fold the operand scale into the (positively homogeneous) PReLU: scale taps and bias
              const float gsc = p0.x * mr1.y, gsh = p0.y - mr1.x * mr1.y * p0.x;
              const float w0 = p0.z * act_s, w1 = p0.w * act_s, w2 = p1.x * act_s, bd = p1.y * act_s;
              // channels past K (K % 32 != 0: the last slab's second half) are rows of the NEXT sample: boundary path, zeroed
              float4 upre;
              if (dw_interior && c < a.K) v[sub][j] = dw_channel<DCLS, true, TRAIN>(q0, q1, q2, gsc, gsh, w0, w1, w2, bd, pslope, first, tstep, tbase, a.frames, true, dls, dlss, &upre);
              else v[sub][j] = dw_channel<DCLS, false, TRAIN>(q0, q1, q2, gsc, gsh, w0, w1, w2, bd, pslope, first, tstep, tbase, a.frames, c < a.K, dls, dlss, &upre);
              if (TRAIN && nt == 0 && c < a.K) {  // the taps carry the operand scale: undo it (power of two, exact)
                const float ia = 1.f / act_s;
                *reinterpret_cast<float4*>(a.dw_u_pre_out + ((size_t)b * a.K + c) * a.pitch + tbase) =
                    make_float4(upre.x * ia, upre.y * ia, upre.z * ia, upre.w * ia);
              }
              dep += v[sub][j].x + (q0.x + q1.x) + (q2.x + p1.y);
            }
          } else {
#pragma unroll
            for (int j = 0; j < CPW; ++j) {
              const int k = ks * KS + sub * RC + pw * CPW + j;
              const uint32_t r0 = rb_s + 4u * (uint32_t)((pw * CPW + j) * TM + lane * 4);
              float4 x = lds128(r0);
              if (PRO == PRO_RES) {
                // x_new = x + rstd2*r + (v1 - mean2*rstd2*v2): the previous block's residual update, applied on the fly;
                // the n-tile-0 item of each time tile also writes x_new for the block after next
                const float4 rr = lds128(r0 + 4u * RC * TM);
                const float cst = s_res[k] - mr_res.x * mr_res.y * s_res[g.k_slabs * KS + k];
                x.x = fmaf(mr_res.y, rr.x, x.x + cst); x.y = fmaf(mr_res.y, rr.y, x.y + cst);
                x.z = fmaf(mr_res.y, rr.z, x.z + cst); x.w = fmaf(mr_res.y, rr.w, x.w + cst);
                if (tbase + 0 >= a.frames) x.x = 0.f;
                if (tbase + 1 >= a.frames) x.y = 0.f;
                if (tbase + 2 >= a.frames) x.z = 0.f;
                if (tbase + 3 >= a.frames) x.w = 0.f;
                if (nt == 0 && k < a.K) *reinterpret_cast<float4*>(a.res_x_out + ((size_t)b * a.K + k) * a.pitch + tbase) = x;
                dep += rr.x + rr.w;
              }
              dep += x.x + x.w;
              if (k >= a.K) x = make_float4(0.f, 0.f, 0.f, 0.f);  // rows past K belong to the next sample
              if (PRO == PRO_PRELU) {
                x.x = prelu_f(x.x, pslope); x.y = prelu_f(x.y, pslope); x.z = prelu_f(x.z, pslope); x.w = prelu_f(x.w, pslope);
              }
              x.x *= act_s; x.y *= act_s; x.z *= act_s; x.w *= act_s;
              v[sub][j] = x;
            }
          }
        }
        // every lane's loads are complete once `dep` exists; then the warp hands both raw slots back
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int sub = 0; sub < SUBS; ++sub) mbar_arrive_after(ptx::smem_u32(&hdr->rempty[rsv[sub]]), dep);
        }
        ptx::mbar_wait(ptx::smem_u32(&hdr->empty[s]), ph ^ 1u);
        const uint32_t ob = op0 + (uint32_t)s * g.op_stage_bytes;
#pragma unroll
        for (int sub = 0; sub < SUBS; ++sub) {
#pragma unroll
          for (int j = 0; j < CPW; ++j) {
            // MN-major 16-bit SWIZZLE_128B: atoms of 64 time steps x 8 channels (1024 B): channel row r = kl & 7 at r*128 B,
            // 16-byte chunks (8 time steps) XOR r; time atoms 1024 B apart (LBO), 8-channel groups 2048 B apart (SBO)
            const int kl = sub * RC + pw * CPW + j;
            const uint32_t r8 = (uint32_t)(kl & 7);
            const uint32_t off16 = (uint32_t)(kl >> 3) * 2048u + (uint32_t)(lane >> 4) * 1024u + r8 * 128u +
                                   (((uint32_t)((lane & 15) >> 1) ^ r8) << 4) + (uint32_t)(lane & 1) * 8u;
            uint2 h2, l2;
            ptx::split_f16x2(v[sub][j].x, v[sub][j].y, h2.x, l2.x);
            ptx::split_f16x2(v[sub][j].z, v[sub][j].w, h2.y, l2.y);
            sts64(ob + off16, h2.x, h2.y);
            sts64(ob + A_BYTES + off16, l2.x, l2.y);
          }
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->full[s]));
        if (++s == g.op_stages) { s = 0; ph ^= 1u; }
      }
      if (PRO == PRO_DW && nt == 0) {
        // the sums were taken over act_s * u: undo the power-of-two scale exactly in double
        const double inv = 1.0 / (double)act_s;
        const double sd = warp_sum_d((double)dls.x + (double)dls.y) * inv, ssd = warp_sum_d((double)dlss.x + (double)dlss.y) * inv * inv;
        if (lane == 0) { atomicAdd(&a.dw_stats_out[2 * b], sd); atomicAdd(&a.dw_stats_out[2 * b + 1], ssd); }
      }
    }
  } else if (warp == 4) {
    // ===================================== MMA ISSUER =======================================================
    int s = 0;
    uint32_t ph = 0;
    const bool leader = ptx::elect_one();
    const uint64_t da_t = ptx::make_smem_desc(0, 1024u, 2048u, 2u);  // A: MN-major SWIZZLE_128B (64-step atoms, 8-channel groups)
    const uint64_t dw_t = ptx::make_smem_desc(0, 16u, 512u, 4u);     // W: K-major SWIZZLE_64B rows of 32 k
    for (int it = 0; it < items_per_cta; ++it) {
      const int acc = it & 1;
      ptx::mbar_wait(ptx::smem_u32(&hdr->tempty[acc]), ((uint32_t)(it >> 1) & 1u) ^ 1u);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
      int prev_s = -1;
      for (int ks = 0; ks < g.k_slabs; ++ks) {
        ptx::mbar_wait(ptx::smem_u32(&hdr->full[s]), ph);
        ptx::tc_fence_after();
        const uint32_t st_base = op0 + (uint32_t)s * g.op_stage_bytes;
        const uint32_t a_hi = st_base >> 4, a_lo = (st_base + A_BYTES) >> 4;
        const uint32_t w_hi = (st_base + 2 * A_BYTES) >> 4, w_lo = w_hi + (g.w_bytes >> 4);
        if (leader) {
#pragma unroll
          for (int kk = 0; kk < KS / 16; ++kk) {
            const uint64_t da_hi = da_t | (uint64_t)(a_hi + kk * 256), dw_hi = dw_t | (uint64_t)(w_hi + kk * 2);
            const uint64_t da_lo = da_t | (uint64_t)(a_lo + kk * 256), dw_lo = dw_t | (uint64_t)(w_lo + kk * 2);
            ptx::mma_f16(d_tmem, da_hi, dw_hi, g.idesc, (ks | kk) ? 1u : 0u);
            if (kk == 0 && prev_s >= 0) ptx::mma_commit(ptx::smem_u32(&hdr->empty[prev_s]));  // previous slab's stage
            ptx::mma_f16(d_tmem, da_lo, dw_hi, g.idesc, 1u);
            ptx::mma_f16(d_tmem, da_hi, dw_lo, g.idesc, 1u);
          }
          if (ks == g.k_slabs - 1) {
            ptx::mma_commit(ptx::smem_u32(&hdr->empty[s]));
            ptx::mma_commit(ptx::smem_u32(&hdr->tfull[acc]));
          }
        }
        __syncwarp();
        prev_s = s;
        if (++s == g.op_stages) { s = 0; ph ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ===================================== EPILOGUE =========================================================
    // thread = one time step (TMEM lane); columns = output channels; TMEM read in 16-column chunks, double buffered
    float eslope = 0.f;
    if (EPI == EPI_H) eslope = a.slope[0];
    const bool store_pre = EPI == EPI_H && a.store_pre != 0;
    float* sp = reinterpret_cast<float*>(smem + SMEM_PARAMS);
    const int egroup = (EGROUPS == 2 && warp >= FIRST_PROD + PROD_WARPS) ? 1 : 0;
    const int te = (warp & 3) * 32 + lane;
    const int tid_e = egroup * 128 + te;
    float2 dacc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) dacc[i] = make_float2(0.f, 0.f);
    for (int it = 0; it < items_per_cta; ++it) {
      int nt, tt, b;
      decode(it, nt, tt, b);
      const int acc = it & 1;
      const int t = tt * TM + te;
      const bool tvalid = t < a.frames;
      const int n0 = nt * g.n_tile;
      const int nvalid = min(g.n_tile, a.M - n0);
      if (EPI == EPI_H || EPI == EPI_MASKDEC) {
        asm volatile("bar.sync 1, %0;" ::"n"(128 * EGROUPS) : "memory");  // previous item's readers are done with sp
        for (int i = tid_e; i < g.n_tile; i += 128 * EGROUPS) sp[i] = i < nvalid ? __ldg(a.bias + n0 + i) : 0.f;
        asm volatile("bar.sync 1, %0;" ::"n"(128 * EGROUPS) : "memory");
      }
      ptx::mbar_wait(ptx::smem_u32(&hdr->tfull[acc]), (uint32_t)(it >> 1) & 1u);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * 256u + ((uint32_t)((warp & 3) * 32) << 16);
      float* Dp = a.D + ((size_t)b * a.M + n0) * a.pitch + t;
      float ls = 0.f, lss = 0.f;
      const int ncols_all = (nvalid + 15) & ~15;
      const int csplit = EGROUPS == 2 ? ((ncols_all / 2 + 15) & ~15) : ncols_all;
      const int cbeg = egroup == 0 ? 0 : csplit;
      const int ncols = egroup == 0 ? csplit : ncols_all;
      // every time step of the tile is a real frame; `tvalid &&` is implied, and stating it keeps the PRO_DW kernels at 122 registers
      const bool tile_full = tvalid && tt * TM + TM <= a.frames;
      // EPI_MASKDEC: w_hat[n][t] = w[n][t] * sigmoid(logit) is contracted on the spot with the decoder basis:
      //   full[8 t + k] += w_hat[n][t] * Dec[n][k], k < 16 (ConvTranspose1d(N,1,16,stride 8), filterbank.py:245-247), 16 partial
      // sums per thread (= per frame) in registers across the n-tiles of one source
      const float* sD = reinterpret_cast<const float*>(raw0_p + (size_t)g.raw_stages * g.raw_stage_bytes);
      float* accbuf = const_cast<float*>(sD) + a.Nb * 16;
      const float* Wp = (EPI == EPI_MASKDEC) ? a.wenc + (size_t)b * a.Nb * a.pitch + t : nullptr;
      const int nb0 = (EPI == EPI_MASKDEC) ? n0 % a.Nb : 0;
      if (EPI == EPI_MASKDEC && nb0 == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dacc[i] = make_float2(0.f, 0.f);
      }
      // the 16 encoder values w[n][t] of a column chunk are fetched one chunk AHEAD of their use (L2 / HBM latency ~700 cycles and
      // only two epilogue warps per scheduler: loading at the point of use left the FMULs below waiting on the scoreboard)
      auto load_w = [&](float (&wv)[16], int c0) {
#pragma unroll
        for (int j = 0; j < 16; ++j) wv[j] = (c0 + j < nvalid) ? __ldg(Wp + (size_t)(nb0 + c0 + j) * a.pitch) : 0.f;
      };
      auto process_dec = [&](const uint32_t (&buf)[16], const float (&wv)[16], int c0) {
        const float osc = ssc_all[n0 + c0];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float logit = fmaf(__uint_as_float(buf[j]), osc, sp[c0 + j]);
          float o = __fdividef(wv[j], 1.f + __expf(-logit));
          if (!tvalid || c0 + j >= nvalid) o = 0.f;
          const float4* dr = reinterpret_cast<const float4*>(sD + (size_t)(nb0 + c0 + j) * 16);
          const float2 o2 = make_float2(o, o);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const float4 d4 = dr[q4];
            dacc[2 * q4] = __ffma2_rn(o2, make_float2(d4.x, d4.y), dacc[2 * q4]);
            dacc[2 * q4 + 1] = __ffma2_rn(o2, make_float2(d4.z, d4.w), dacc[2 * q4 + 1]);
          }
        }
      };
      auto process = [&](const uint32_t (&buf)[16], const float (&wv)[16], int c0) {
        if (EPI == EPI_MASKDEC) { process_dec(buf, wv, c0); return; }
        float* q = Dp + (size_t)c0 * a.pitch;
        const bool full = (c0 + 16 <= nvalid) && tile_full;  // warp-uniform
        const float osc = ssc_all[n0 + c0];  // one power-of-two scale per 16-row weight group (and the operand scale)
        float o[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          float pvv[4] = {0.f, 0.f, 0.f, 0.f};
          if (EPI == EPI_H) {
            const float4 p4 = *reinterpret_cast<const float4*>(sp + c0 + j4 * 4);
            pvv[0] = p4.x; pvv[1] = p4.y; pvv[2] = p4.z; pvv[3] = p4.w;
          }
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int j = j4 * 4 + jj;
            float v = __uint_as_float(buf[j]);
            if (EPI == EPI_RAW) v *= osc;
            if (EPI == EPI_H) {
              const float pre = fmaf(v, osc, pvv[jj]);
              const float act = prelu_f(pre, eslope);
              v = store_pre ? pre : act;
              if (full) { ls += act; lss = fmaf(act, act, lss); }
            }
            o[j] = v;
          }
        }
        if (full) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            *q = o[j];
            q += a.pitch;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float v = tvalid ? o[j] : 0.f;
            if (c0 + j < nvalid) {
              q[(size_t)j * a.pitch] = v;
              if (EPI == EPI_H) { const float sv = store_pre ? prelu_f(v, eslope) : v; ls += sv; lss = fmaf(sv, sv, lss); }
            }
          }
        }
      };
      uint32_t bufA[16], bufB[16];
      float wvA[16], wvB[16];
      if (EPI == EPI_MASKDEC && cbeg < ncols) load_w(wvA, cbeg);
      if (cbeg < ncols) ptx::tmem_ld16(taddr + (uint32_t)cbeg, bufA);
      for (int c0 = cbeg; c0 < ncols; c0 += 32) {
        ptx::tmem_ld_wait();
        if (c0 + 16 < ncols) {
          ptx::tmem_ld16(taddr + (uint32_t)(c0 + 16), bufB);
          if (EPI == EPI_MASKDEC) load_w(wvB, c0 + 16);
        }
        process(bufA, wvA, c0);
        ptx::tmem_ld_wait();
        if (c0 + 32 < ncols) {
          ptx::tmem_ld16(taddr + (uint32_t)(c0 + 32), bufA);
          if (EPI == EPI_MASKDEC) load_w(wvA, c0 + 32);
        }
        if (c0 + 16 < ncols) process(bufB, wvB, c0 + 16);
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(ptx::smem_u32(&hdr->tempty[acc]));
      if (EPI == EPI_MASKDEC && (n0 + g.n_tile) % a.Nb == 0) {
        // last n-tile of source s: combine the two column halves (epilogue groups) and the two overlapping frames, crop
        // (conv_tasnet.py:169) and store.  Thread (group gq, frame te) owns samples 8 te + 4 gq .. +3 of the tile.
        float4* ab = reinterpret_cast<float4*>(accbuf + ((size_t)egroup * 128 + te) * 16);
        ab[0] = make_float4(dacc[0].x, dacc[0].y, dacc[1].x, dacc[1].y);
        ab[1] = make_float4(dacc[2].x, dacc[2].y, dacc[3].x, dacc[3].y);
        ab[2] = make_float4(dacc[4].x, dacc[4].y, dacc[5].x, dacc[5].y);
        ab[3] = make_float4(dacc[6].x, dacc[6].y, dacc[7].x, dacc[7].y);
        asm volatile("bar.sync 1, %0;" ::"n"(128 * EGROUPS) : "memory");
        const int src = n0 / a.Nb, S = a.M / a.Nb;
        float* yo = a.D + ((size_t)b * S + src) * (size_t)a.dec_T_out;
        const float4 c0a = *reinterpret_cast<const float4*>(accbuf + (size_t)te * 16 + egroup * 4);
        const float4 c0b = *reinterpret_cast<const float4*>(accbuf + (size_t)(128 + te) * 16 + egroup * 4);
        float4 v = make_float4(c0a.x + c0b.x, c0a.y + c0b.y, c0a.z + c0b.z, c0a.w + c0b.w);
        if (te > 0) {
          const float4 p0 = *reinterpret_cast<const float4*>(accbuf + (size_t)(te - 1) * 16 + 8 + egroup * 4);
          const float4 p1 = *reinterpret_cast<const float4*>(accbuf + (size_t)(128 + te - 1) * 16 + 8 + egroup * 4);
          v.x += p0.x + p1.x; v.y += p0.y + p1.y; v.z += p0.z + p1.z; v.w += p0.w + p1.w;
        }
        const long long tau = (long long)8 * t + egroup * 4 - a.dec_crop_left;
        const float vv[4] = {v.x, v.y, v.z, v.w};
        if (te > 0 && tau >= 0 && tau + 3 < a.dec_T_out && ((reinterpret_cast<uintptr_t>(yo + tau) & 15) == 0)) {
          *reinterpret_cast<float4*>(yo + tau) = v;
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (tau + e < 0 || tau + e >= a.dec_T_out) continue;
            if (te > 0) yo[tau + e] = vv[e];
            else atomicAdd(yo + tau + e, vv[e]);   // first frame of the tile: the previous tile's last frame adds its taps 8..15
          }
        }
        if (te == 127) {  // taps 8..15 of the tile's last frame land in the next tile's first 8 samples
          const float4 q0 = *reinterpret_cast<const float4*>(accbuf + (size_t)127 * 16 + 8 + egroup * 4);
          const float4 q1 = *reinterpret_cast<const float4*>(accbuf + (size_t)(128 + 127) * 16 + 8 + egroup * 4);
          const float tv[4] = {q0.x + q1.x, q0.y + q1.y, q0.z + q1.z, q0.w + q1.w};
          const long long tau2 = (long long)8 * (t + 1) + egroup * 4 - a.dec_crop_left;
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (tau2 + e >= 0 && tau2 + e < a.dec_T_out) atomicAdd(yo + tau2 + e, tv[e]);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(128 * EGROUPS) : "memory");  // accbuf is reused by the next source
      }
      if (EPI == EPI_H) {
        const double sd = warp_sum_d((double)ls), ssd = warp_sum_d((double)lss);
        if (lane == 0) { atomicAdd(&a.stats_out[2 * b], sd); atomicAdd(&a.stats_out[2 * b + 1], ssd); }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (warp == 4) ptx::tmem_dealloc(tmem_base, 512);
}

// ---- host side ----------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D fp32 map over a (rows, pitch) activation tensor; box = box_rows x box_cols; out-of-bounds elements read as zero
int make_map(CUtensorMap* tm, const float* ptr, int rows, int pitch, int box_cols, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return CTN_ENOTBUILT;
  const cuuint64_t gdim[2] = {(cuuint64_t)pitch, (cuuint64_t)rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)pitch * 4};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? CTN_OK : CTN_EINVAL;
}

template <int PRO, int EPI, int DWM = 0>
int launch(const TmaArgs& g, size_t smem, int grid, cudaStream_t st) {
  static bool attr_done[CTN_MAX_DEVICES] = {false};
  const int dev = ctn_current_device();
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_pw_tma<PRO, EPI, DWM>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr_done[dev] = true;
  }
  k_pw_tma<PRO, EPI, DWM><<<grid, Roles<PRO>::THREADS, smem, st>>>(g);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

}  // namespace

// 1 when (pro, epi, shape) is served by the TMA-fed kernels (fp16-piece mode only); the caller falls back to k_pw_umma otherwise
int ctn_pw_tma_supported(const PwArgs& a, int pro, int epi) {
  if (!encode_fn() || eff_math(a.M, CTN_MATH_F16X3) != CTN_MATH_F16X3) return 0;  // fp16 weight images only
  if (!((pro == PRO_DW && epi == EPI_RAW) || ((pro == PRO_RES || pro == PRO_NONE) && epi == EPI_H) || (pro == PRO_PRELU && epi == EPI_MASKDEC)))
    return 0;
  if (epi == EPI_MASKDEC) {
    const int n_tile = pick_n_tile(a.M);
    if (!a.dec_w || a.Nb <= 0 || a.M % a.Nb != 0 || a.Nb % n_tile != 0 || a.Nb > 1024) return 0;  // whole n-tiles per source; basis fits smem
  }
  if (a.pitch % TM != 0) return 0;
  if ((a.dw_in_slope != nullptr) != (a.dw_u_pre_out != nullptr)) return 0;
  if (pro == PRO_DW && (a.dw_pad_left != a.dw_dilation || a.dw_dilation < 1 || !a.dw_params ||
                        !(a.dw_dilation == 1 || a.dw_dilation == 2 || a.dw_dilation % 4 == 0)))
    return 0;
  return 1;
}

int ctn_pw_tma(const PwArgs& a, int pro, int epi, cudaStream_t st) {
  if (!a.wimg) return CTN_EINVAL;
  if ((((uintptr_t)a.A) | ((uintptr_t)a.wimg)) & 15) return CTN_EALIGN;
  TmaArgs g;
  memset(&g, 0, sizeof(g));
  g.a = a;
  g.n_tile = pick_n_tile(a.M);
  g.n_tiles = (a.M + g.n_tile - 1) / g.n_tile;
  g.k_slabs = (a.K + KS - 1) / KS;
  g.t_tiles = a.pitch / TM;
  g.num_items = a.B * g.t_tiles * g.n_tiles;
  g.w_bytes = (uint32_t)g.n_tile * (uint32_t)(KS * 2);
  g.wimg = reinterpret_cast<const uint8_t*>(a.wimg);
  g.oscale = reinterpret_cast<const float*>(g.wimg + (size_t)g.n_tiles * g.k_slabs * 2 * g.n_tile * KS * sizeof(__half));
  g.act_scale = a.act_scale;
  g.dwp = a.dw_params;
  g.idesc = ptx::make_idesc_f16(TM, g.n_tile, /*A MN-major*/ 1, /*B K-major*/ 0);
  // header: barriers + epilogue parameters (HDR_FIXED), the output scale table, then (PRO_RES) the folded bias vectors v1, v2 of the
  // previous block for all K channels (two global loads per channel and stage sat on the producers' critical path otherwise)
  g.res_tab_off = (uint32_t)(HDR_FIXED + g.n_tiles * g.n_tile * 4);
  g.reverse = pro == PRO_DW;
  g.hdr_bytes = (uint32_t)((g.res_tab_off + (pro == PRO_RES ? 2 * g.k_slabs * KS * 4 : 0) + 1023) & ~1023u);
  g.op_stage_bytes = 2u * A_BYTES + 2u * g.w_bytes;
  uint32_t raw_data = 0;
  if (pro == PRO_DW) {
    const int d = a.dw_dilation;
    g.dw_three = 2 * ((d + 3) & ~3) + TM > 256;  // the TMA box is at most 256 elements wide
    g.dw_pad = g.dw_three ? 0 : ((d + 3) & ~3);
    raw_data = g.dw_three ? 3u * RC * TM * 4 : (uint32_t)(RC * (TM + 2 * g.dw_pad) * 4);
    g.raw_tx_bytes = raw_data + RC * 32;
    CTN_TRY(make_map(&g.tmA, a.A, a.B * a.K, a.pitch, g.dw_three ? TM : TM + 2 * g.dw_pad, RC));
  } else {
    raw_data = (pro == PRO_RES ? 2u : 1u) * RC * TM * 4;
    g.raw_tx_bytes = raw_data;
    CTN_TRY(make_map(&g.tmA, a.A, a.B * a.K, a.pitch, TM, RC));
    if (pro == PRO_RES) CTN_TRY(make_map(&g.tmR, a.res_r, a.B * a.res_Mt, a.pitch, TM, RC));
  }
  g.raw_stage_bytes = (g.raw_tx_bytes + 1023u) & ~1023u;
  const size_t dec_bytes = epi == EPI_MASKDEC ? ((size_t)a.Nb * 16 + 2 * 128 * 16) * sizeof(float) : 0;
  const size_t budget = 227 * 1024 - 1024 - g.hdr_bytes - dec_bytes;
  // 3 operand stages (fewer if they do not fit), then as many raw stages as fit
  int op = 3;
  while (op > 2 && (size_t)op * g.op_stage_bytes + 2 * (size_t)g.raw_stage_bytes > budget) --op;
  if ((size_t)op * g.op_stage_bytes + 2 * (size_t)g.raw_stage_bytes > budget) return CTN_EUNSUPPORTED;
  int raw = (int)((budget - (size_t)op * g.op_stage_bytes) / g.raw_stage_bytes);
  if (raw > MAX_RAW) raw = MAX_RAW;
  g.op_stages = op;
  g.raw_stages = raw;
  const size_t smem = 1024 + g.hdr_bytes + (size_t)op * g.op_stage_bytes + (size_t)raw * g.raw_stage_bytes + dec_bytes;
  int grid = ctn_num_sms();
  if (grid > g.num_items) grid = g.num_items;
  if (pro == PRO_DW && epi == EPI_RAW) {
    if (a.dw_in_slope) {  // training forward
      if (g.dw_three) return launch<PRO_DW, EPI_RAW, 8 | 4>(g, smem, grid, st);
      if (a.dw_dilation >= 4) return launch<PRO_DW, EPI_RAW, 8 | 3>(g, smem, grid, st);
      return a.dw_dilation == 2 ? launch<PRO_DW, EPI_RAW, 8 | 2>(g, smem, grid, st) : launch<PRO_DW, EPI_RAW, 8 | 1>(g, smem, grid, st);
    }
    if (g.dw_three) return launch<PRO_DW, EPI_RAW, 4>(g, smem, grid, st);
    if (a.dw_dilation >= 4) return launch<PRO_DW, EPI_RAW, 3>(g, smem, grid, st);
    return a.dw_dilation == 2 ? launch<PRO_DW, EPI_RAW, 2>(g, smem, grid, st) : launch<PRO_DW, EPI_RAW, 1>(g, smem, grid, st);
  }
  if (pro == PRO_RES && epi == EPI_H) return launch<PRO_RES, EPI_H>(g, smem, grid, st);
  if (pro == PRO_NONE && epi == EPI_H) return launch<PRO_NONE, EPI_H>(g, smem, grid, st);
  if (pro == PRO_PRELU && epi == EPI_MASKDEC) {
    const int tiles = a.B * g.t_tiles;
    return launch<PRO_PRELU, EPI_MASKDEC>(g, smem, grid < tiles ? grid : tiles, st);
  }
  return CTN_EUNSUPPORTED;
}
