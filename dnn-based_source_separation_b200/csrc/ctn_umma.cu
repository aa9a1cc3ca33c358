// tcgen05 (5th-gen tensor core) implementation of the dense 1x1 "pointwise" contractions of the Conv-TasNet path.
//
//   D[b][n][t] = epi( sum_k W[n][k] * pro(A[b][k][t]) )        A: (B,K,pitch) fp32, time contiguous
//
// Orientation: TIME runs along the UMMA M dimension (TMEM lanes), output channels along N (TMEM columns):
//   * the activation operand is consumed as an MN-major (time-contiguous) SWIZZLE_128B_BASE32B shared-memory tile, i.e. the
//     (channels, time) tensor is used as it lies in HBM -- no transposition anywhere;
//   * the weight operand is K-major (PyTorch (out,in,1) layout), pre-arranged once per forward into the exact
//     swizzled shared-memory image so that one 1-D bulk async copy (TMA engine) brings a 32-channel slab in;
//   * the epilogue reads a TMEM lane = one time step per thread, so every global store of a warp is a contiguous
//     128-byte row segment of D.
// fp32-parity numerics: x = hi + lo with 11-bit pieces, D = A_hi W_hi + A_lo W_hi + A_hi W_lo accumulated in fp32 in TMEM
// (the dropped lo*lo term is ~2^-22 relative).  Pieces are TF32 ("3xTF32", kind::tf32) or FP16 ("3xFP16", kind::f16: twice
// the tensor rate, half the shared memory per stage; weights pre-scaled per 16-row group, see wimg_f16_group) -- template
// parameter F16.  The layouts described here are the TF32 ones; the FP16 ones are next to the code that stages them.
//
// One persistent CTA per SM, warp-specialised:
//   warps 0-3   epilogue  (TMEM -> registers -> fused epilogue -> coalesced global stores)
//   warp  4     TMEM allocator + single-thread tcgen05.mma issuer
//   warps 5-12  producers (global -> registers -> prologue + hi/lo split -> swizzled st.shared; one thread also issues
//               the bulk copies of the weight slabs)
// Pipelines: smem ring (full/empty mbarriers, tcgen05.commit frees a stage) and a 2-deep TMEM accumulator ring.
#include "ctn_internal.h"
#include "ctn_umma_ptx.cuh"
#include "ctn_dw_math.cuh"
#include <cuda_fp16.h>

namespace {

constexpr int TM = 128;       // time steps per tile (UMMA M)
#ifndef CTN_KS
#define CTN_KS 32
#endif
constexpr int KS = CTN_KS;    // input channels per smem slab.  32: 128-byte weight rows (SWIZZLE_128B), 2-3 stages;
                              // 16: 64-byte rows (SWIZZLE_64B), 4-6 stages -- measured SLOWER (per-slab handshakes dominate)
constexpr int A_BYTES = TM * KS * 4;  // 8 KB per precision
constexpr int MAX_STAGES = 8;
constexpr uint32_t W_LAYOUT = KS == 32 ? 2u : 4u;    // UMMA layout type of the weight operand (SWIZZLE_128B / SWIZZLE_64B)
constexpr uint32_t W_SBO = KS == 32 ? 1024u : 512u;  // bytes between 8-row groups of the weight image
constexpr int NUM_THREADS_DW = 21 * 32;   // PRO_DW kernels: 4 epilogue + 1 MMA + 16 producer warps (2 channels each)
constexpr int NUM_THREADS_E8 = 17 * 32;   // other kernels: 4 + 1 + 8 producer warps + a second epilogue warpgroup (13-16)
constexpr int SMEM_HEADER = 2048 + CTN_F16_MAX_ROWS * 4;  // barriers + tmem pointer, the epilogue parameter row, the fp16-mode output scales
constexpr int SMEM_SCALES = 2048;   // byte offset of float[CTN_F16_MAX_ROWS]: power-of-two scale of every padded output channel of the
                                    // contraction (F16 kernels), loaded ONCE per CTA (a per-item staging put a global-load latency
                                    // on the epilogue's critical path: +0.9 us per item, 0.5 ms per step)
constexpr int SMEM_PARAMS = 1024;   // byte offset of float[256] inside the header

struct UmmaArgs {
  PwArgs a;
  const float* wimg;  // [n_tiles][k_slabs][NPASS][n_tile*32] swizzled images
  const float* oscale;  // fp16-piece mode: [n_tiles*n_tile] per-output-channel scale 2^-e (stored behind the images)
  int n_tile, n_tiles, k_slabs, t_tiles, num_items, stages;
  uint32_t stage_bytes, w_bytes;  // w_bytes: bytes per precision of a weight slab (n_tile*128)
  uint32_t idesc, lbo_a, sbo_a, lbo_w, sbo_w, a_layout, w_layout;
};

// producer warps per prologue: the depthwise producer always runs 16; the residual-update producer (pw1, the second
// largest kernel, latency-bound: 47 % issue-active) can run 8 or 16 -- compile-time switch CTN_RES_WARPS16
#ifndef CTN_RES_WARPS16
#define CTN_RES_WARPS16 0  // measured: 16 warps (72 registers) 3.66 ms vs 3.28 ms with 8 warps (96 registers) at cfg2
#endif
template <int PRO> struct Roles {
  static constexpr int PROD_WARPS = (PRO == PRO_DW || (PRO == PRO_RES && CTN_RES_WARPS16)) ? 16 : 8;
  static constexpr int EGROUPS = PRO == PRO_DW ? 1 : 2;
  static constexpr int THREADS = (4 + 1 + PROD_WARPS + 4 * (EGROUPS - 1)) * 32;
};
static_assert(Roles<PRO_DW>::THREADS == NUM_THREADS_DW && Roles<PRO_NONE>::THREADS == NUM_THREADS_E8, "role layout");

struct __align__(8) SmemHeader {
  uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
  uint64_t tfull[2];
  uint64_t tempty[2];
  uint32_t tmem_base;
};

template <int DCLS, bool INTERIOR, int CPW>
__device__ __forceinline__ void dw_slab(const PwArgs& a, int b, int ks, int pw, int tbase, float2 mr1, float pslope,
                                        bool prefetch_next, float4 (&v)[CPW], float2& dls, float2& dlss) {
  const int d = a.dw_dilation, pl = a.dw_pad_left;
  const int step = DCLS == 4 ? d : 4;
  const int first = DCLS == 4 ? tbase - pl : tbase - 4;
  float4 q[CPW][3];
  float pg[CPW], pb[CPW], pbd[CPW], pw0[CPW], pw1[CPW], pw2[CPW];
#pragma unroll
  for (int j = 0; j < CPW; ++j) {
    const int c = ks * KS + pw * CPW + j;
    const int cc = INTERIOR ? c : (c < a.K ? c : a.K - 1);
    const float* hr = a.A + ((size_t)b * a.K + cc) * a.pitch;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      int ts = first + k * step;
      if (!INTERIOR) ts = ts < 0 ? 0 : (ts > a.pitch - 4 ? a.pitch - 4 : ts);
      q[j][k] = __ldg(reinterpret_cast<const float4*>(hr + ts));
    }
    pg[j] = __ldg(a.dw_norm_g + cc); pb[j] = __ldg(a.dw_norm_b + cc); pbd[j] = __ldg(a.dw_b + cc);
    pw0[j] = __ldg(a.dw_w + cc * 3); pw1[j] = __ldg(a.dw_w + cc * 3 + 1); pw2[j] = __ldg(a.dw_w + cc * 3 + 2);
  }
  if (prefetch_next && INTERIOR) {
    // pull the next slab's rows towards the SM while this slab is being computed (no register cost)
#pragma unroll
    for (int j = 0; j < CPW; ++j) {
      const float* hr = a.A + ((size_t)b * a.K + (ks + 1) * KS + pw * CPW + j) * a.pitch;
#pragma unroll
      for (int k = 0; k < 3; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(hr + first + k * step));
    }
  }
#pragma unroll
  for (int j = 0; j < CPW; ++j) {
    const int c = ks * KS + pw * CPW + j;
    const float gsc = pg[j] * mr1.y, gsh = pb[j] - mr1.x * mr1.y * pg[j];
    v[j] = dw_channel<DCLS, INTERIOR>(q[j][0], q[j][1], q[j][2], gsc, gsh, pw0[j], pw1[j], pw2[j], pbd[j], pslope, first, step,
                                      tbase, a.frames, c < a.K, dls, dlss);
  }
}

// F16: operands are staged as fp16 hi/lo pieces (kind::f16, "3xFP16"): A MN-major SWIZZLE_128B (atoms of 64 time steps x 8
// channels), W K-major SWIZZLE_64B (rows of 32 channels = 64 bytes) -- both pinned on hardware by tools/umma_unit_f16.cu.
// Half the shared-memory bytes per stage (4-deep ring at N = 256) and half the tensor-pipe time of the TF32 split.
template <int PRO, int EPI, int NPASS, bool F16>
__global__ void __launch_bounds__(Roles<PRO>::THREADS, 1) k_pw_umma(const UmmaArgs g) {
  constexpr int NPREC = NPASS == 3 ? 2 : 1;  // precisions staged per operand (hi [, lo])
  constexpr int A_BYTES = F16 ? TM * KS * 2 : TM * KS * 4;  // bytes of one precision of the activation slab (shadows the tf32 constant)
  static_assert(!F16 || NPASS == 3, "fp16 operands: 3-pass split");
  constexpr int EGROUPS = Roles<PRO>::EGROUPS;  // epilogue warpgroups (each covers all 128 TMEM lanes)
  constexpr int PROD_WARPS = Roles<PRO>::PROD_WARPS;
  constexpr int CPW = KS / PROD_WARPS;            // channels of a slab per producer warp (2 or 4)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;  // SWIZZLE_128B atoms need 1024-byte alignment
  uint8_t* smem = smem_raw + (base - raw);
  SmemHeader* hdr = reinterpret_cast<SmemHeader*>(smem);
  const uint32_t stage0 = base + SMEM_HEADER;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const PwArgs& a = g.a;

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.stages; ++s) {
      ptx::mbar_init(ptx::smem_u32(&hdr->full[s]), PROD_WARPS + 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->empty[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(ptx::smem_u32(&hdr->tfull[i]), 1);
      ptx::mbar_init(ptx::smem_u32(&hdr->tempty[i]), 128 * EGROUPS);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 4) ptx::tmem_alloc(ptx::smem_u32(&hdr->tmem_base), 512);
  // fp16 pieces: power-of-two scale of the activation operand (|operand| * act_s <= 2^15 by construction, ctn_act_scales),
  // undone together with the weight-group scales in the epilogue
  float act_s = 1.f;
  if constexpr (F16) {
    if (a.act_scale) act_s = __ldg(a.act_scale);
    const float inv = 1.f / act_s;
    float* ssc_all = reinterpret_cast<float*>(smem + SMEM_SCALES);
    for (int i = threadIdx.x; i < g.n_tiles * g.n_tile; i += blockDim.x) ssc_all[i] = __ldg(g.oscale + i) * inv;
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = hdr->tmem_base;

  // Work decomposition: CTA c walks the items J = c + it * gridDim.x; J -> (weight tile nt = J % n_tiles, time tile
  // L = J / n_tiles -> (b, tt)).  n-tile fastest: co-running CTAs read the same activations while they are in L2.
  const int items_per_cta = (g.num_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  auto decode = [&](int it2, int& nt2, int& tt2, int& b2) {
    const int J = (int)blockIdx.x + it2 * (int)gridDim.x;
    nt2 = J % g.n_tiles;
    const int L = J / g.n_tiles;
    tt2 = L % g.t_tiles;
    b2 = L / g.t_tiles;
  };

  if (warp >= 5 && warp < 5 + PROD_WARPS) {
    // ===================================== PRODUCERS ========================================================
    const int p = threadIdx.x - 160;  // 0 .. 32*PROD_WARPS-1
    const int pw = p >> 5;            // producer warp: rows pw*CPW .. pw*CPW+CPW-1 of the slab
    float pslope = 0.f;
    if (PRO == PRO_PRELU || PRO == PRO_DW) pslope = a.pro_slope[0];
    int s = 0;
    uint32_t ph = 0;
    // activation loads of slab (it2, ks2): issued ONE SLAB AHEAD of their use (register double buffer), across item
    // boundaries, so that the global-load latency overlaps the split/store work and the barrier waits
    auto load_A = [&](int it2, int ks2, float4 (&dst)[CPW], float4 (&dstr)[CPW]) {
      int nt2, tt2, b2;
      decode(it2, nt2, tt2, b2);
      const float* Ab2 = a.A + (size_t)b2 * a.K * a.pitch + (size_t)tt2 * TM + lane * 4;
#pragma unroll
      for (int j = 0; j < CPW; ++j) {
        const int k = ks2 * KS + pw * CPW + j;
        dst[j] = k < a.K ? __ldg(reinterpret_cast<const float4*>(Ab2 + (size_t)k * a.pitch)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (PRO == PRO_RES) {
        const float* Rb2 = a.res_r + (size_t)b2 * a.res_Mt * a.pitch + (size_t)tt2 * TM + lane * 4;
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int k = ks2 * KS + pw * CPW + j;
          dstr[j] = k < a.K ? __ldg(reinterpret_cast<const float4*>(Rb2 + (size_t)k * a.pitch)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    float4 vnext[CPW], rnext[CPW];
    if (PRO != PRO_DW && items_per_cta > 0) load_A(0, 0, vnext, rnext);
    for (int it = 0; it < items_per_cta; ++it) {
      int nt, tt, b;
      decode(it, nt, tt, b);
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(g.wimg) + (size_t)nt * g.k_slabs * NPREC * g.w_bytes;
      // PRO_DW: per-sample gLN1 statistics of h (the A operand)
      float2 mr1 = make_float2(0.f, 1.f);
      float2 dls = make_float2(0.f, 0.f), dlss = make_float2(0.f, 0.f);
      if (PRO == PRO_DW) mr1 = gln_mean_rstd(a.dw_stats_in + 2 * b, (double)a.K * (double)a.frames, a.dw_eps);
      float2 mr_res = make_float2(0.f, 1.f);
      if (PRO == PRO_RES) mr_res = gln_mean_rstd(a.res_stats + 2 * b, a.res_n, a.res_eps);
      const int tbase = tt * TM + lane * 4;  // first of this thread's 4 time steps
      int dcls = 4;
      bool dw_interior = false;
      if (PRO == PRO_DW) {
        const int d = a.dw_dilation;
        dcls = d >= 4 ? 4 : d;
        const int reach = d >= 4 ? d : 4;  // furthest sample touched on either side of the tile
        dw_interior = (tt * TM - reach >= 0) && (tt * TM + TM - 1 + reach + 3 < a.frames) && (a.K % KS == 0) &&
                      (a.dw_pad_left == d);
      }
      for (int ks = 0; ks < g.k_slabs; ++ks) {
        float4 v[CPW];
        if (PRO != PRO_DW) {
#pragma unroll
          for (int j = 0; j < CPW; ++j) v[j] = vnext[j];
          if (PRO == PRO_RES) {
            // x_new = x + rstd2*r + (v1 - mean2*rstd2*v2): the previous block's residual update, applied on the fly;
            // the n-tile-0 CTA of each time tile also writes x_new for the block after next
#pragma unroll
            for (int j = 0; j < CPW; ++j) {
              const int k = ks * KS + pw * CPW + j;
              const int kc = k < a.K ? k : a.K - 1;
              const float cst = __ldg(a.res_v1 + kc) - mr_res.x * mr_res.y * __ldg(a.res_v2 + kc);
              float4 xn;
              xn.x = fmaf(mr_res.y, rnext[j].x, v[j].x + cst); xn.y = fmaf(mr_res.y, rnext[j].y, v[j].y + cst);
              xn.z = fmaf(mr_res.y, rnext[j].z, v[j].z + cst); xn.w = fmaf(mr_res.y, rnext[j].w, v[j].w + cst);
              if (tbase + 0 >= a.frames) xn.x = 0.f;
              if (tbase + 1 >= a.frames) xn.y = 0.f;
              if (tbase + 2 >= a.frames) xn.z = 0.f;
              if (tbase + 3 >= a.frames) xn.w = 0.f;
              if (k >= a.K) xn = make_float4(0.f, 0.f, 0.f, 0.f);
              v[j] = xn;
              if (nt == 0 && k < a.K)
                *reinterpret_cast<float4*>(a.res_x_out + ((size_t)b * a.K + k) * a.pitch + tbase) = xn;
            }
          }
          const int ks_n = ks + 1 < g.k_slabs ? ks + 1 : 0;
          const int it_n = ks + 1 < g.k_slabs ? it : it + 1;
          if (it_n < items_per_cta) load_A(it_n, ks_n, vnext, rnext);
        } else {
          // u[c][t] = PReLU( sum_k wd[c][k] * hn[c][t + k*d - pl] + bd[c] ), hn = gLN1(h) inside [0,frames), 0 outside.
          // All 12 128-bit loads of the slab (4 channels x 3 taps) are issued before any arithmetic.  The branch below is
          // uniform over the CTA (depends on the item only).
          const bool pfn = ks + 1 < g.k_slabs;
          if (dw_interior) {
            if (dcls == 4) dw_slab<4, true, CPW>(a, b, ks, pw, tbase, mr1, pslope, pfn, v, dls, dlss);
            else if (dcls == 2) dw_slab<2, true, CPW>(a, b, ks, pw, tbase, mr1, pslope, pfn, v, dls, dlss);
            else dw_slab<1, true, CPW>(a, b, ks, pw, tbase, mr1, pslope, pfn, v, dls, dlss);
          } else {
            if (dcls == 4) dw_slab<4, false, CPW>(a, b, ks, pw, tbase, mr1, pslope, pfn, v, dls, dlss);
            else if (dcls == 2) dw_slab<2, false, CPW>(a, b, ks, pw, tbase, mr1, pslope, pfn, v, dls, dlss);
            else dw_slab<1, false, CPW>(a, b, ks, pw, tbase, mr1, pslope, pfn, v, dls, dlss);
          }
        }
        ptx::mbar_wait(ptx::smem_u32(&hdr->empty[s]), ph ^ 1u);
        const uint32_t st_base = stage0 + (uint32_t)s * g.stage_bytes;
        if (p == 0) {
          const uint32_t fb = ptx::smem_u32(&hdr->full[s]);
          ptx::mbar_arrive_expect_tx(fb, NPREC * g.w_bytes);
          ptx::bulk_g2s(st_base + NPREC * A_BYTES, wsrc + (size_t)ks * NPREC * g.w_bytes, NPREC * g.w_bytes, fb);
        }
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int kl = pw * CPW + j;  // 0..KS-1 within the slab
          const int kg = kl >> 2, r = kl & 3;
          // MN-major tf32 needs SWIZZLE_128B_BASE32B (the only MN-major layout the tensor core accepts for 32-bit
          // operands; pinned on hardware with tools/umma_unit.cu): atoms of 4 channel rows x 128 B (32 time steps),
          // 32-byte chunks XOR (row & 3); atoms along time 512 B apart (LBO), 4-channel groups 2048 B apart (SBO).
          const uint32_t off = (uint32_t)kg * 2048u + (uint32_t)(lane >> 3) * 512u + (uint32_t)r * 128u +
                               (uint32_t)(((((lane & 7) >> 1) ^ r) << 5) | ((lane & 1) << 4));
          float4 x = v[j];
          if (PRO == PRO_PRELU) {
            x.x = prelu_f(x.x, pslope); x.y = prelu_f(x.y, pslope); x.z = prelu_f(x.z, pslope); x.w = prelu_f(x.w, pslope);
          }
          if constexpr (F16) {
            x.x *= act_s; x.y *= act_s; x.z *= act_s; x.w *= act_s;
            // MN-major 16-bit SWIZZLE_128B: atoms of 64 time steps x 8 channels (1024 B): channel row r = kl & 7 at r*128 B,
            // 16-byte chunks (8 time steps) XOR r; time atoms 1024 B apart (LBO), 8-channel groups 2048 B apart (SBO)
            const uint32_t r8 = (uint32_t)(kl & 7);
            const uint32_t off16 = (uint32_t)(kl >> 3) * 2048u + (uint32_t)(lane >> 4) * 1024u + r8 * 128u +
                                   (((uint32_t)((lane & 15) >> 1) ^ r8) << 4) + (uint32_t)(lane & 1) * 8u;
            uint2 h2, l2;
            ptx::split_f16x2(x.x, x.y, h2.x, l2.x);
            ptx::split_f16x2(x.z, x.w, h2.y, l2.y);
            *reinterpret_cast<uint2*>(smem + SMEM_HEADER + (size_t)s * g.stage_bytes + off16) = h2;
            *reinterpret_cast<uint2*>(smem + SMEM_HEADER + (size_t)s * g.stage_bytes + A_BYTES + off16) = l2;
          } else {
          float4 hi, lo;
          hi.x = ptx::hi_tf32(x.x); hi.y = ptx::hi_tf32(x.y); hi.z = ptx::hi_tf32(x.z); hi.w = ptx::hi_tf32(x.w);
          {  // lo = x - hi (exact), two elements per FADD2
            const float2 l01 = __fadd2_rn(make_float2(x.x, x.y), make_float2(-hi.x, -hi.y));
            const float2 l23 = __fadd2_rn(make_float2(x.z, x.w), make_float2(-hi.z, -hi.w));
            lo = make_float4(l01.x, l01.y, l23.x, l23.y);
          }
          *reinterpret_cast<float4*>(smem + SMEM_HEADER + (size_t)s * g.stage_bytes + off) = hi;
          if (NPASS == 3) *reinterpret_cast<float4*>(smem + SMEM_HEADER + (size_t)s * g.stage_bytes + A_BYTES + off) = lo;
          }
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->full[s]));
        if (++s == g.stages) { s = 0; ph ^= 1u; }
      }
      if (PRO == PRO_DW && nt == 0) {
        const double sd = warp_sum_d((double)dls.x + (double)dls.y), ssd = warp_sum_d((double)dlss.x + (double)dlss.y);
        if (lane == 0) { atomicAdd(&a.dw_stats_out[2 * b], sd); atomicAdd(&a.dw_stats_out[2 * b + 1], ssd); }
      }
    }
  } else if (warp == 4) {
    // ===================================== MMA ISSUER =======================================================
    // The whole warp walks the loop converged; one elected lane issues.  The stage-free commit of slab q is issued
    // AFTER the first MMA of slab q+1 (same item), so the tensor pipe always has work queued while the thread is busy
    // with the commit / barrier bookkeeping.
    int s = 0;
    uint32_t ph = 0;
    const bool leader = ptx::elect_one();
    // descriptor templates: only the 14-bit start-address field changes
    const uint64_t da_t = ptx::make_smem_desc(0, g.lbo_a, g.sbo_a, g.a_layout);
    const uint64_t dw_t = ptx::make_smem_desc(0, g.lbo_w, g.sbo_w, g.w_layout);
    for (int it = 0; it < items_per_cta; ++it) {
      const int acc = it & 1;
      ptx::mbar_wait(ptx::smem_u32(&hdr->tempty[acc]), ((uint32_t)(it >> 1) & 1u) ^ 1u);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
      int prev_s = -1;
      for (int ks = 0; ks < g.k_slabs; ++ks) {
        ptx::mbar_wait(ptx::smem_u32(&hdr->full[s]), ph);
        ptx::tc_fence_after();
        const uint32_t st_base = stage0 + (uint32_t)s * g.stage_bytes;
        const uint32_t a_hi = st_base >> 4, a_lo = (st_base + A_BYTES) >> 4;
        const uint32_t w_hi = (st_base + NPREC * A_BYTES) >> 4, w_lo = w_hi + (g.w_bytes >> 4);
        if (leader) {
          auto mma = [&](uint64_t da, uint64_t dw, uint32_t accum) {
            if constexpr (F16) ptx::mma_f16(d_tmem, da, dw, g.idesc, accum);
            else ptx::mma_tf32(d_tmem, da, dw, g.idesc, accum);
          };
#pragma unroll
          // per instruction: 8 channels (tf32) or 16 (fp16); either way the A start address advances by 4096 B (two channel
          // groups) and the W start address by 32 B
          for (int kk = 0; kk < (F16 ? KS / 16 : KS / 8); ++kk) {
            const uint64_t da_hi = da_t | (uint64_t)(a_hi + kk * 256), dw_hi = dw_t | (uint64_t)(w_hi + kk * 2);
            mma(da_hi, dw_hi, (ks | kk) ? 1u : 0u);
            if (kk == 0 && prev_s >= 0) ptx::mma_commit(ptx::smem_u32(&hdr->empty[prev_s]));  // previous slab's stage (its MMAs are queued ahead)
            if (NPASS == 3) {
              const uint64_t da_lo = da_t | (uint64_t)(a_lo + kk * 256), dw_lo = dw_t | (uint64_t)(w_lo + kk * 2);
              mma(da_lo, dw_hi, 1u);
              mma(da_hi, dw_lo, 1u);
            }
          }
          if (ks == g.k_slabs - 1) {
            ptx::mma_commit(ptx::smem_u32(&hdr->empty[s]));     // last slab of the item: free its stage right away
            ptx::mma_commit(ptx::smem_u32(&hdr->tfull[acc]));   // accumulator ready for the epilogue
          }
        }
        __syncwarp();
        prev_s = s;
        if (++s == g.stages) { s = 0; ph ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ===================================== EPILOGUE =========================================================
    // thread = one time step (TMEM lane); columns = output channels.  Per-channel parameters of the tile are staged
    // in shared memory once per item; TMEM is read in 16-column chunks, double buffered so that the next tcgen05.ld is
    // in flight while the current chunk is transformed and stored (one coalesced 128-byte row segment per warp-store).
    float eslope = 0.f;
    if (EPI == EPI_H) eslope = a.slope[0];
    const bool store_pre = EPI == EPI_H && a.store_pre != 0;  // training forward: keep the PRE-activation, statistics of PReLU(.)
    float* sp = reinterpret_cast<float*>(smem + SMEM_PARAMS);  // [256] per-channel epilogue parameter
    const int egroup = (EGROUPS == 2 && warp >= 5 + PROD_WARPS) ? 1 : 0;                     // second warpgroup handles the upper half of the columns
    const int te = (warp & 3) * 32 + lane;                     // time step within the tile == TMEM lane
    const int tid_e = egroup * 128 + te;
    for (int it = 0; it < items_per_cta; ++it) {
      int nt, tt, b;
      decode(it, nt, tt, b);
      const int acc = it & 1;
      const int t = tt * TM + te;
      const bool tvalid = t < a.frames;
      const int n0 = nt * g.n_tile;
      const int nvalid = min(g.n_tile, a.M - n0);
      float mscale = 1.f;
      {
        // stage the per-channel parameter: EPI_HEAD: v1 - mean*rstd*v2 (deferred gLN shift); EPI_H / EPI_MASK: bias
        float2 mr = make_float2(0.f, 1.f);
        if (EPI == EPI_HEAD) { mr = gln_mean_rstd(a.stats_in + 2 * b, a.n_in, a.eps); mscale = mr.y; }
        asm volatile("bar.sync 1, %0;" ::"n"(128 * EGROUPS) : "memory");  // previous item's readers are done with sp
        for (int i = tid_e; i < g.n_tile; i += 128 * EGROUPS) {
          float pv = 0.f;
          if (i < nvalid) {
            if (EPI == EPI_HEAD) pv = __ldg(a.v1 + n0 + i) - mr.x * mr.y * __ldg(a.v2 + n0 + i);
            if (EPI == EPI_H || EPI == EPI_MASK) pv = __ldg(a.bias + n0 + i);
          }
          sp[i] = pv;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(128 * EGROUPS) : "memory");
      }
      ptx::mbar_wait(ptx::smem_u32(&hdr->tfull[acc]), (uint32_t)(it >> 1) & 1u);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * 256u + ((uint32_t)((warp & 3) * 32) << 16);
      float* Dp = a.D + ((size_t)b * a.M + n0) * a.pitch + t;
      float* Mp = (EPI == EPI_MASK && a.mask_out) ? a.mask_out + ((size_t)b * a.M + n0) * a.pitch + t : nullptr;
      const float* Wp = (EPI == EPI_MASK) ? a.wenc + (size_t)b * a.Nb * a.pitch + t : nullptr;
      const int nb0 = (EPI == EPI_MASK) ? n0 % a.Nb : 0;
      float ls = 0.f, lss = 0.f;
      const int ncols_all = (nvalid + 15) & ~15;
      const int csplit = EGROUPS == 2 ? ((ncols_all / 2 + 15) & ~15) : ncols_all;  // group 0: [0,csplit), group 1: rest
      const int cbeg = egroup == 0 ? 0 : csplit;
      const int ncols = egroup == 0 ? csplit : ncols_all;

      const bool tile_full = tt * TM + TM <= a.frames;  // every time step of this tile is a real frame
      auto process = [&](const uint32_t (&buf)[16], int c0) {
        float wv[16];
        if (EPI == EPI_MASK) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            int nn = nb0 + c0 + j;
            while (nn >= a.Nb) nn -= a.Nb;
            wv[j] = (c0 + j < nvalid) ? __ldg(Wp + (size_t)nn * a.pitch) : 0.f;
          }
        }
        float* q = Dp + (size_t)c0 * a.pitch;
        float* qm = Mp ? Mp + (size_t)c0 * a.pitch : nullptr;
        const bool full = (c0 + 16 <= nvalid) && tile_full;  // warp-uniform
        // F16: the 16 output channels of a chunk share one power-of-two weight scale (wimg_f16_rows scales 16-row groups)
        float osc = 1.f;
        if constexpr (F16) osc = reinterpret_cast<const float*>(smem + SMEM_SCALES)[n0 + c0];
        float o[16], mk[16];
        // per-channel parameters are fetched 4 columns at a time (8 live registers instead of 32: the epilogue shares the
        // register budget of the producers)
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 p4 = *reinterpret_cast<const float4*>(sp + c0 + j4 * 4);
          const float pvv[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int j = j4 * 4 + jj;
            float v = __uint_as_float(buf[j]);
            mk[j] = 0.f;
            // F16: v * osc undoes the power-of-two row scaling of the weights (exact), folded into the bias FMA
            if (EPI == EPI_RAW && F16) v *= osc;
            if (EPI == EPI_HEAD) v = F16 ? fmaf(mscale * osc, v, pvv[jj]) : fmaf(mscale, v, pvv[jj]);
            if (EPI == EPI_H) {
              const float pre = F16 ? fmaf(v, osc, pvv[jj]) : v + pvv[jj];
              const float act = prelu_f(pre, eslope);
              v = store_pre ? pre : act;
              if (full) { ls += act; lss = fmaf(act, act, lss); }  // gLN statistics are always those of PReLU(.)
            }
            if (EPI == EPI_MASK) {
              const float logit = F16 ? fmaf(v, osc, pvv[jj]) : v + pvv[jj];
              if (a.mask_logits) {  // softmax masks: the normalisation over all S*N channels is a second pass (ctn_softmax_mask)
                mk[j] = logit;
                v = logit;
              } else {
                mk[j] = __fdividef(1.f, 1.f + __expf(-logit));
                v = mk[j] * wv[j];
              }
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
          if (EPI == EPI_MASK && qm) {
#pragma unroll
            for (int j = 0; j < 16; ++j) { *qm = mk[j]; qm += a.pitch; }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float v = tvalid ? o[j] : 0.f;
            if (c0 + j < nvalid) {
              q[(size_t)j * a.pitch] = v;
              if (EPI == EPI_MASK && qm) qm[(size_t)j * a.pitch] = tvalid ? mk[j] : 0.f;
              if (EPI == EPI_H) { const float sv = store_pre ? prelu_f(v, eslope) : v; ls += sv; lss = fmaf(sv, sv, lss); }
            }
          }
        }
      };

      uint32_t bufA[16], bufB[16];
      if (cbeg < ncols) ptx::tmem_ld16(taddr + (uint32_t)cbeg, bufA);
      for (int c0 = cbeg; c0 < ncols; c0 += 32) {
        ptx::tmem_ld_wait();
        if (c0 + 16 < ncols) ptx::tmem_ld16(taddr + (uint32_t)(c0 + 16), bufB);
        process(bufA, c0);
        ptx::tmem_ld_wait();
        if (c0 + 32 < ncols) ptx::tmem_ld16(taddr + (uint32_t)(c0 + 32), bufA);
        if (c0 + 16 < ncols) process(bufB, c0 + 16);
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(ptx::smem_u32(&hdr->tempty[acc]));
      if (EPI == EPI_H) {
        double s = warp_sum_d((double)ls), ss = warp_sum_d((double)lss);
        if (lane == 0) { atomicAdd(&a.stats_out[2 * b], s); atomicAdd(&a.stats_out[2 * b + 1], ss); }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (warp == 4) ptx::tmem_dealloc(tmem_base, 512);
}

// ---- weight images ---------------------------------------------------------------------------------------------
// K-major SWIZZLE_64B image of an (n_tile x KS=16) weight slab: rows of 64 B (16 k), 8-row groups of 512 B (SBO),
// 16-byte chunk index XOR ((row >> 1) & 3).  Float offset of element (row nl, k kl):
__host__ __device__ __forceinline__ int wimg_offset(int nl, int kl) {
  if (KS == 32)  // SWIZZLE_128B: rows of 128 B, 8-row groups of 1024 B, chunk index XOR (row & 7)
    return (nl >> 3) * 256 + (nl & 7) * 32 + ((((kl >> 2) ^ (nl & 7)) << 2) | (kl & 3));
  return (nl >> 3) * 128 + (nl & 7) * 16 + ((((kl >> 2) ^ ((nl >> 1) & 3)) << 2) | (kl & 3));
}

// grid (k_slabs, n_tiles), block 256: builds the image(s) of one weight slab.
__global__ void __launch_bounds__(256) k_build_wimg(const float* __restrict__ W, int M, int K, int n_tile, int k_slabs,
                                                    int nprec, float* __restrict__ wimg) {
  const int ks = blockIdx.x, nt = blockIdx.y;
  const size_t per = (size_t)n_tile * KS;  // floats per precision
  float* dst = wimg + ((size_t)nt * k_slabs + ks) * nprec * per;
  for (int i = threadIdx.x; i < n_tile * KS; i += 256) {
    const int nl = i / KS, kl = i % KS;
    const int n = nt * n_tile + nl, k = ks * KS + kl;
    const float x = (n < M && k < K) ? W[(size_t)n * K + k] : 0.f;
    const int off = wimg_offset(nl, kl);
    const float hi = ptx::to_tf32(x);
    dst[off] = hi;
    if (nprec == 2) dst[per + off] = ptx::to_tf32(x - hi);
  }
}

// fp16 variant ("3xFP16"): K-major SWIZZLE_64B rows of 32 k x 2 B; per slab a hi image then a lo image of n_tile*64 bytes.
// Every group of 16 weight ROWS (output channels) is first scaled by a power of two 2^e so that its largest entry lands in
// [2^9, 2^10) (one scale per 16 rows = per 16-column epilogue chunk, so the epilogue needs a single scalar per chunk):
// hi and lo pieces then sit in fp16's normal range whatever the magnitude of the weights (tiny gamma-folded rows would
// otherwise lose their lo piece to fp16's subnormal floor of 6e-8, huge ones would saturate); the epilogue multiplies the
// accumulator of channel n by the exact inverse 2^-e (oscale, stored behind the images).
// One warp per row; block = 16 warps = one 16-row scale group (the epilogue reads one scale per 16-column chunk);
// grid (ceil(n_tile/16), n_tiles).
__device__ __forceinline__ void wimg_f16_group(const float* __restrict__ W, int M, int K, int n_tile, int k_slabs, int nt, int grp,
                                               __half* __restrict__ img, float* __restrict__ oscale, float* smax) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nl = grp * 16 + wid;
  const int n = nt * n_tile + nl;
  const bool live = nl < n_tile && n < M;
  const float* row = W + (size_t)n * K;
  float mx = 0.f;
  if (live)
    for (int k = lane; k < K; k += 32) mx = fmaxf(mx, fabsf(row[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) smax[wid] = mx;
  __syncthreads();
  mx = smax[lane & 15];
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  __syncthreads();  // smax is reused by the next group of this block
  int e = 0;
  if (mx > 0.f && mx < INFINITY) e = 9 - ilogbf(mx);  // 2^e * (largest entry of the 16 rows) in [2^9, 2^10)
  e = max(-100, min(100, e));
  const float up = ldexpf(1.f, e), down = ldexpf(1.f, -e);
  if (nl >= n_tile) return;
  if (lane == 0) oscale[n] = down;
  const size_t per = (size_t)n_tile * KS;  // halves per precision
  for (int ks = 0; ks < k_slabs; ++ks) {
    const int kl = lane, k = ks * KS + kl;  // KS == 32 == warp size
    const float x = (live && k < K) ? row[k] * up : 0.f;
    __half* dst = img + ((size_t)nt * k_slabs + ks) * 2 * per;
    const int off = (nl >> 3) * 256 + (nl & 7) * 32 + ((((kl >> 3) ^ ((nl >> 1) & 3))) << 3) + (kl & 7);  // in halves
    const __half hi = __float2half_rn(x);
    dst[off] = hi;
    dst[per + off] = __float2half_rn(x - __half2float(hi));
  }
}
__host__ __device__ inline size_t wimg_f16_image_bytes(int n_tile, int n_tiles, int k_slabs) {
  return (size_t)n_tiles * k_slabs * 2 * n_tile * KS * sizeof(__half);
}
__global__ void __launch_bounds__(512) k_build_wimg_f16(const float* __restrict__ W, int M, int K, int n_tile, int k_slabs,
                                                        int n_tiles, float* __restrict__ wimg) {
  static_assert(KS == 32, "one lane per channel of a slab");
  __shared__ float smax[16];
  __half* img = reinterpret_cast<__half*>(wimg);
  float* oscale = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(wimg) + wimg_f16_image_bytes(n_tile, n_tiles, k_slabs));
  wimg_f16_group(W, M, K, n_tile, k_slabs, blockIdx.y, blockIdx.x, img, oscale, smax);
}

struct WimgJobs { WimgJob j[CTN_MAX_JOBS]; };
// grid (max k_slabs * max n_tiles, jobs): one block per (slab, n-tile) of one job
__global__ void __launch_bounds__(256) k_build_wimg_batch(const WimgJobs jobs, int nprec) {
  const WimgJob& jb = jobs.j[blockIdx.y];
  const int n_tile = pick_n_tile(jb.M);
  const int n_tiles = (jb.M + n_tile - 1) / n_tile, k_slabs = (jb.K + KS - 1) / KS;
  const size_t per = (size_t)n_tile * KS;
  for (int blk = blockIdx.x; blk < n_tiles * k_slabs; blk += gridDim.x) {
    const int nt = blk / k_slabs, ks = blk - nt * k_slabs;
    float* dst = jb.wimg + ((size_t)nt * k_slabs + ks) * nprec * per;
    for (int i = threadIdx.x; i < n_tile * KS; i += 256) {
      const int nl = i / KS, kl = i % KS;
      const int n = nt * n_tile + nl, k = ks * KS + kl;
      const float x = (n < jb.M && k < jb.K) ? jb.W[(size_t)n * jb.K + k] : 0.f;
      const int off = wimg_offset(nl, kl);
      const float hi = ptx::to_tf32(x);
      dst[off] = hi;
      if (nprec == 2) dst[per + off] = ptx::to_tf32(x - hi);
    }
  }
}

// grid (64, jobs), block 512: blockIdx.x walks the (n-tile, 16-row group) pairs of its job
__global__ void __launch_bounds__(512) k_build_wimg_batch_f16(const WimgJobs jobs) {
  __shared__ float smax[16];
  const WimgJob& jb = jobs.j[blockIdx.y];
  const int n_tile = pick_n_tile(jb.M);
  const int n_tiles = (jb.M + n_tile - 1) / n_tile, k_slabs = (jb.K + KS - 1) / KS;
  const int groups = n_tile / 16;
  __half* img = reinterpret_cast<__half*>(jb.wimg);
  float* oscale = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(jb.wimg) + wimg_f16_image_bytes(n_tile, n_tiles, k_slabs));
  for (int blk = blockIdx.x; blk < n_tiles * groups; blk += gridDim.x)
    wimg_f16_group(jb.W, jb.M, jb.K, n_tile, k_slabs, blk / groups, blk % groups, img, oscale, smax);
}

template <int PRO, int EPI, int NPASS, bool F16>
int launch(const UmmaArgs& g, size_t smem, int grid, cudaStream_t st) {
  static bool attr_done[CTN_MAX_DEVICES] = {false};  // the opt-in is per device (context)
  const int dev = ctn_current_device();
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_pw_umma<PRO, EPI, NPASS, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr_done[dev] = true;
  }
  k_pw_umma<PRO, EPI, NPASS, F16><<<grid, Roles<PRO>::THREADS, smem, st>>>(g);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

}  // namespace

extern "C" int ctn_has_tcgen05(void) { return 1; }

size_t ctn_umma_wimg_bytes(int M, int K, int math) {
  const int nprec = math == CTN_MATH_TF32 ? 1 : 2;
  const int n_tile = pick_n_tile(M);
  const int n_tiles = (M + n_tile - 1) / n_tile, k_slabs = (K + KS - 1) / KS;
  // fp16 images are half the size but carry the per-channel scale array behind them; the tf32x3 size + scales covers both
  return (size_t)n_tiles * k_slabs * nprec * n_tile * KS * sizeof(float) + (size_t)n_tiles * n_tile * sizeof(float) + 256;
}

int ctn_umma_build_wimg(const float* W, int M, int K, int math, float* wimg, cudaStream_t st) {
  math = eff_math(M, math);
  const int nprec = math == CTN_MATH_TF32 ? 1 : 2;  // hi [, lo]
  const int n_tile = pick_n_tile(M);
  const int n_tiles = (M + n_tile - 1) / n_tile, k_slabs = (K + KS - 1) / KS;
  if (math == CTN_MATH_F16X3) {
    k_build_wimg_f16<<<dim3(n_tile / 16, n_tiles), 512, 0, st>>>(W, M, K, n_tile, k_slabs, n_tiles, wimg);
    CTN_COUNT_LAUNCH();
    CTN_RETURN_IF_CUDA_ERR();
    return CTN_OK;
  }
  k_build_wimg<<<dim3(k_slabs, n_tiles), 256, 0, st>>>(W, M, K, n_tile, k_slabs, nprec, wimg);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

int ctn_umma_build_wimg_batch(const WimgJob* jobs, int n, int math, cudaStream_t st) {
  const int nprec = math == CTN_MATH_TF32 ? 1 : 2;
  bool uniform = true;
  for (int i = 0; i < n; ++i) uniform = uniform && eff_math(jobs[i].M, math) == math;
  if (!uniform) {  // some jobs fall back to the tf32 pieces (eff_math): per-job launches
    for (int i = 0; i < n; ++i) CTN_TRY(ctn_umma_build_wimg(jobs[i].W, jobs[i].M, jobs[i].K, math, jobs[i].wimg, st));
    return CTN_OK;
  }
  for (int i0 = 0; i0 < n; i0 += CTN_MAX_JOBS) {
    WimgJobs wj;
    const int m = n - i0 < CTN_MAX_JOBS ? n - i0 : CTN_MAX_JOBS;
    int maxb = 1;
    for (int i = 0; i < m; ++i) {
      wj.j[i] = jobs[i0 + i];
      const int n_tile = pick_n_tile(jobs[i0 + i].M);
      const int blocks = ((jobs[i0 + i].M + n_tile - 1) / n_tile) * ((jobs[i0 + i].K + KS - 1) / KS);
      if (blocks > maxb) maxb = blocks;
    }
    if (math == CTN_MATH_F16X3) k_build_wimg_batch_f16<<<dim3(64, m), 512, 0, st>>>(wj);
    else k_build_wimg_batch<<<dim3(maxb, m), 256, 0, st>>>(wj, nprec);
    CTN_COUNT_LAUNCH();
  }
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

int ctn_pw_umma(const PwArgs& a, int pro, int epi, int math, cudaStream_t st) {
  if (!a.wimg) return CTN_EINVAL;
  math = eff_math(a.M, math);
  if (a.pitch % TM != 0) return CTN_EALIGN;
  if ((((uintptr_t)a.A) | ((uintptr_t)a.wimg)) & 15) return CTN_EALIGN;
  UmmaArgs g;
  g.a = a;
  g.wimg = a.wimg;
  g.n_tile = pick_n_tile(a.M);
  g.n_tiles = (a.M + g.n_tile - 1) / g.n_tile;
  g.k_slabs = (a.K + KS - 1) / KS;
  g.t_tiles = a.pitch / TM;
  g.num_items = a.B * g.t_tiles * g.n_tiles;
  const int nprec = math == CTN_MATH_TF32 ? 1 : 2;
  const bool f16 = math == CTN_MATH_F16X3;
  const uint32_t a_bytes = f16 ? (uint32_t)(TM * KS * 2) : (uint32_t)A_BYTES;
  g.w_bytes = (uint32_t)g.n_tile * (uint32_t)(KS * (f16 ? 2 : 4));
  g.stage_bytes = (uint32_t)nprec * (a_bytes + g.w_bytes);
  const size_t budget = 227 * 1024 - SMEM_HEADER - 1024;
  int stages = (int)(budget / g.stage_bytes);
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  if (stages < 1) return CTN_EUNSUPPORTED;
  g.stages = stages;
  g.oscale = nullptr;
  if (f16) {
    g.oscale = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(a.wimg) + wimg_f16_image_bytes(g.n_tile, g.n_tiles, g.k_slabs));
    g.idesc = ptx::make_idesc_f16(TM, g.n_tile, /*A MN-major*/ 1, /*B K-major*/ 0);
    g.lbo_a = 1024u; g.sbo_a = 2048u; g.a_layout = 2u;  // 64-time-step atoms adjacent, 8-channel groups 2048 B apart
    g.lbo_w = 16u; g.sbo_w = 512u; g.w_layout = 4u;      // SWIZZLE_64B rows of 32 k
  } else {
    g.idesc = ptx::make_idesc_tf32(TM, g.n_tile, /*A MN-major*/ 1, /*B K-major*/ 0);
    g.lbo_a = 512u;   // between 32-time-step atoms
    g.sbo_a = 2048u;  // between 4-channel groups
    g.lbo_w = 16u;    // unused for swizzled K-major
    g.sbo_w = W_SBO;  // between 8-row (output channel) groups
    g.a_layout = 1u; g.w_layout = W_LAYOUT;
  }
  const size_t smem = SMEM_HEADER + 1024 + (size_t)stages * g.stage_bytes;
  int grid = ctn_num_sms();
  if (grid > g.num_items) grid = g.num_items;
#define UM_LAUNCH(P, E)                                                                                     \
  if (pro == P && epi == E)                                                                                 \
    return f16 ? launch<P, E, 3, true>(g, smem, grid, st)                                                   \
               : (nprec == 2 ? launch<P, E, 3, false>(g, smem, grid, st) : launch<P, E, 1, false>(g, smem, grid, st));
  UM_LAUNCH(PRO_NONE, EPI_RAW)
  UM_LAUNCH(PRO_DW, EPI_RAW)
  UM_LAUNCH(PRO_NONE, EPI_HEAD)
  UM_LAUNCH(PRO_NONE, EPI_H)
  UM_LAUNCH(PRO_RES, EPI_H)
  UM_LAUNCH(PRO_PRELU, EPI_MASK)
#undef UM_LAUNCH
  return CTN_EUNSUPPORTED;
}
