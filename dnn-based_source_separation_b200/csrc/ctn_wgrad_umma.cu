// tcgen05 weight-gradient kernel of the 1x1 convolutions (training path):
//
//   dW[m][k] += sum_b sum_{t < frames} dY[b][m][t] * X[b][k][t]            dY: (B, M, pitch), X: (B, K, pitch)
//
// Both operands are reduced over TIME, which is the contiguous dimension of both tensors, so both are K-major UMMA
// operands in the canonical SWIZZLE_128B layout (rows of 32 time steps = 128 bytes): output channels m on the UMMA M
// dimension (TMEM lanes), input channels k on N (TMEM columns), 32 time steps per pipeline stage (4 MMAs of K = 8).
// The reduction over B * frames (128 k at cfg2) is split across the CTAs of a tile ("split-K"): grid = tiles x splits
// ~ one CTA per SM; every CTA accumulates its share of the time axis in ONE TMEM accumulator and adds the tile to dW
// with fp32 reductions at the end (dW must be zero on entry).
// fp32-parity numerics: the same 3xTF32 split as the forward kernels, applied to BOTH operands by the producer warps
// (hi = x rounded to 10 mantissa bits, lo = x - hi exact; D += hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM).
//
// Warp roles (672 threads): warps 0-3 epilogue (idle until the end), warp 4 TMEM allocator + MMA issuer, warps 5-20
// producers in two groups that take alternate stages (global 128-bit loads -> split -> swizzled st.shared; a warp moves
// 4 rows x 128 B per instruction; the loads of a group's next stage are in flight for two stage periods).
#include "ctn_internal.h"
#include "ctn_umma_ptx.cuh"
#include <string.h>

namespace {

constexpr int WG_THREADS = 21 * 32;
constexpr int WG_PW = 16;            // producer warps
constexpr int WG_KT = 32;            // time steps per stage
constexpr int WG_A_BYTES = 128 * 128;  // 128 rows x 128 B per precision
constexpr int WG_HEADER = 1024;
constexpr int WG_MAX_STAGES = 4;

struct WgArgs {
  const float* dy; size_t dy_bs;
  const float* x; size_t x_bs;
  float* dWa; float* dWb; int split_row;  // rows [0, split_row) -> dWa, rows [split_row, M) -> dWb (both (rows, K) row-major)
  int M, K, B, frames, pitch;
  int n_tile, tiles_n, tiles, steps_per_split, chunks, stages;
  uint32_t stage_bytes, idesc, tmem_cols;
};

struct __align__(8) WgHeader {
  uint64_t full[WG_MAX_STAGES];
  uint64_t empty[WG_MAX_STAGES];
  uint64_t done;
  uint32_t tmem_base;
};

template <int NPASS>
__global__ void __launch_bounds__(WG_THREADS, 1) k_wgrad_umma(const WgArgs g) {
  constexpr int NPREC = NPASS == 3 ? 2 : 1;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  WgHeader* hdr = reinterpret_cast<WgHeader*>(smem);
  const uint32_t stage0 = base + WG_HEADER;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int tile = (int)blockIdx.x % g.tiles, split = (int)blockIdx.x / g.tiles;
  const int m0 = (tile / g.tiles_n) * 128, n0 = (tile % g.tiles_n) * g.n_tile;
  const long long total = (long long)g.B * g.chunks;
  const long long s0 = (long long)split * g.steps_per_split;
  const long long s1 = s0 + g.steps_per_split < total ? s0 + g.steps_per_split : total;
  const int nsteps = (int)(s1 - s0);
  if (nsteps <= 0) return;  // uniform over the CTA

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.stages; ++s) {
      ptx::mbar_init(ptx::smem_u32(&hdr->full[s]), WG_PW / 2);  // one group of 8 producer warps fills a stage
      ptx::mbar_init(ptx::smem_u32(&hdr->empty[s]), 1);
    }
    ptx::mbar_init(ptx::smem_u32(&hdr->done), 1);
    ptx::fence_mbar_init();
  }
  if (warp == 4) ptx::tmem_alloc(ptx::smem_u32(&hdr->tmem_base), g.tmem_cols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = hdr->tmem_base;
  const uint32_t b_off = NPREC * WG_A_BYTES;           // B operand (hi) inside a stage
  const uint32_t b_lo_off = b_off + g.n_tile * 128u;   // B operand (lo)

  if (warp >= 5) {
    // ===================================== PRODUCERS ========================================================
    // Two groups of 8 warps take alternate steps (group = step parity): a warp issues the loads of its NEXT step right
    // after storing the current one, two step periods before they are needed, so the global-load latency (1.5-3 us
    // under load: 128-byte row segments) hides behind a full extra step without a second register buffer.
    const int pw = warp - 5;
    const int grp = pw & 1, pwl = pw >> 1;   // group, warp within the group (0..7)
    const int r4 = lane >> 3, ch = lane & 7;
    // row groups of this warp in a step: gi = pwl + 8*i, i < 4 -> dY rows (gi < 32), i >= 4 -> X rows; rows advance by 32
    // per i, so global offsets advance by 32*pitch and shared-memory offsets by 4096 bytes (row & 7 is invariant)
    const int rowA = pwl * 4 + r4;                       // first dY row of this lane (i = 0)
    const uint32_t sw = (uint32_t)(rowA & 7);
    const uint32_t offA0 = (uint32_t)(rowA >> 3) * 1024u + sw * 128u + (uint32_t)((ch ^ sw) << 4);
    const uint32_t offB0 = b_off + offA0;                // same lane pattern inside the X operand
    const int nB = g.n_tile / 32;                        // X row groups of 32 rows per step (<= 8)
    constexpr int NG = 12;                               // 4 dY + up to 8 X groups of 32 rows
    auto load = [&](long long step, float4 (&v)[NG]) {
      const int b = (int)(step / g.chunks), t0 = (int)(step % g.chunks) * WG_KT;
      const int t = t0 + ch * 4;
      const float* pa = g.dy + (size_t)b * g.dy_bs + (size_t)(m0 + rowA) * g.pitch + t;
      const float* pb = g.x + (size_t)b * g.x_bs + (size_t)(n0 + rowA) * g.pitch + t;
      // NOTE: nothing here may READ the loaded values (not even a predicated-off select): that would wait for the data at
      // the load site and serialise the global-load latency into every step (measured: 60 % of the stall samples).
      // Columns at or beyond `frames` are masked where the values are consumed.
#pragma unroll
      for (int i = 0; i < NG; ++i) {
        const bool isA = i < 4;
        const int j = isA ? i : i - 4;
        const bool ok = isA ? (m0 + rowA + 32 * j < g.M) : (j < nB && n0 + rowA + 32 * j < g.K);
        v[i] = ok ? __ldg(reinterpret_cast<const float4*>((isA ? pa : pb) + (size_t)(32 * j) * g.pitch))
                  : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // L2 prefetch, 512 bytes per row at a time: a step reads only 128 B of each of its 384 rows (16 KB apart), which the
    // DRAM serves at ~25 % of its peak (measured 1.6 TB/s).  Every 4th step, lanes 0-3 of each row ask L2 for the four
    // lines of steps it+4 .. it+7 of that row in one burst (same DRAM page); the later 128-bit loads then hit L2.
    auto prefetch = [&](long long step) {
      if (ch >= 4) return;
      const long long sp = step + ch;
      if (sp >= s1) return;
      const int b = (int)(sp / g.chunks), t0 = (int)(sp % g.chunks) * WG_KT;
      const float* pa = g.dy + (size_t)b * g.dy_bs + (size_t)(m0 + rowA) * g.pitch + t0;
      const float* pb = g.x + (size_t)b * g.x_bs + (size_t)(n0 + rowA) * g.pitch + t0;
#pragma unroll
      for (int i = 0; i < NG; ++i) {
        const bool isA = i < 4;
        const int j = isA ? i : i - 4;
        const bool ok = isA ? (m0 + rowA + 32 * j < g.M) : (j < nB && n0 + rowA + 32 * j < g.K);
        if (ok) asm volatile("prefetch.global.L2 [%0];" ::"l"((isA ? pa : pb) + (size_t)(32 * j) * g.pitch));
      }
    };
    static_assert(WG_KT * 4 == 128, "one step of a row is one 128-byte line");
    float4 cur[NG];
    if (grp == 0) prefetch(s0 + 2);
    if (grp < nsteps) load(s0 + grp, cur);
    for (int it = grp; it < nsteps; it += 2) {
      const int s = it % g.stages;
      const uint32_t ph = (uint32_t)(it / g.stages) & 1u;
      ptx::mbar_wait(ptx::smem_u32(&hdr->empty[s]), ph ^ 1u);
      uint8_t* st = smem + WG_HEADER + (size_t)s * g.stage_bytes;
      const int tcol = (int)((s0 + it) % g.chunks) * WG_KT + ch * 4;
      const bool tail = tcol + 3 >= g.frames;
#pragma unroll
      for (int i = 0; i < NG; ++i) {
        const bool isA = i < 4;
        const int j = isA ? i : i - 4;
        if (isA || j < nB) {
          float4 x = cur[i];
          if (tail) {  // pad columns never contribute (last chunk of a sample only)
            if (tcol + 0 >= g.frames) x.x = 0.f;
            if (tcol + 1 >= g.frames) x.y = 0.f;
            if (tcol + 2 >= g.frames) x.z = 0.f;
            if (tcol + 3 >= g.frames) x.w = 0.f;
          }
          float4 hi, lo;
          hi.x = ptx::hi_tf32(x.x); hi.y = ptx::hi_tf32(x.y); hi.z = ptx::hi_tf32(x.z); hi.w = ptx::hi_tf32(x.w);
          const uint32_t off = (isA ? offA0 : offB0) + (uint32_t)j * 4096u;
          *reinterpret_cast<float4*>(st + off) = hi;
          if (NPASS == 3) {
            lo.x = x.x - hi.x; lo.y = x.y - hi.y; lo.z = x.z - hi.z; lo.w = x.w - hi.w;
            // the lo plane of an operand sits right behind its hi plane
            *reinterpret_cast<float4*>(st + off + (isA ? (uint32_t)WG_A_BYTES : g.n_tile * 128u)) = lo;
          }
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&hdr->full[s]));
      if (grp == 0 && (it & 3) == 0) prefetch(s0 + it + 6);  // lines of steps it+6 .. it+9
      if (it + 2 < nsteps) load(s0 + it + 2, cur);
    }
  } else if (warp == 4) {
    // ===================================== MMA ISSUER =======================================================
    int s = 0;
    uint32_t ph = 0;
    const bool leader = ptx::elect_one();
    const uint64_t d_t = ptx::make_smem_desc(0, 16u, 1024u, 2);  // K-major SWIZZLE_128B, 8-row groups 1024 B apart
    for (int it = 0; it < nsteps; ++it) {
      ptx::mbar_wait(ptx::smem_u32(&hdr->full[s]), ph);
      ptx::tc_fence_after();
      const uint32_t st = stage0 + (uint32_t)s * g.stage_bytes;
      const uint32_t a_hi = st >> 4, a_lo = (st + WG_A_BYTES) >> 4;
      const uint32_t b_hi = (st + b_off) >> 4, b_lo = (st + b_lo_off) >> 4;
      if (leader) {
#pragma unroll
        for (int kk = 0; kk < WG_KT / 8; ++kk) {
          const uint64_t da_hi = d_t | (uint64_t)(a_hi + kk * 2), db_hi = d_t | (uint64_t)(b_hi + kk * 2);
          ptx::mma_tf32(tmem_base, da_hi, db_hi, g.idesc, (it | kk) ? 1u : 0u);
          if (NPASS == 3) {
            const uint64_t da_lo = d_t | (uint64_t)(a_lo + kk * 2), db_lo = d_t | (uint64_t)(b_lo + kk * 2);
            ptx::mma_tf32(tmem_base, da_lo, db_hi, g.idesc, 1u);
            ptx::mma_tf32(tmem_base, da_hi, db_lo, g.idesc, 1u);
          }
        }
        ptx::mma_commit(ptx::smem_u32(&hdr->empty[s]));
        if (it == nsteps - 1) ptx::mma_commit(ptx::smem_u32(&hdr->done));
      }
      __syncwarp();
      if (++s == g.stages) { s = 0; ph ^= 1u; }
    }
  } else {
    // ===================================== EPILOGUE =========================================================
    ptx::mbar_wait(ptx::smem_u32(&hdr->done), 0u);
    ptx::tc_fence_after();
    const int m = m0 + warp * 32 + lane;
    float* row = nullptr;
    if (m < g.M) row = m < g.split_row ? g.dWa + (size_t)m * g.K : g.dWb + (size_t)(m - g.split_row) * g.K;
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
    for (int c0 = 0; c0 < g.n_tile; c0 += 16) {
      uint32_t v[16];
      ptx::tmem_ld16(taddr + (uint32_t)c0, v);
      ptx::tmem_ld_wait();
      if (row != nullptr) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int n = n0 + c0 + j;
          if (n < g.K) atomicAdd(row + n, __uint_as_float(v[j]));
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (warp == 4) ptx::tmem_dealloc(tmem_base, g.tmem_cols);
}

template <int NPASS>
int launch_wg(const WgArgs& g, size_t smem, int grid, cudaStream_t st) {
  static bool attr_done[CTN_MAX_DEVICES] = {false};  // the opt-in is per device (context)
  const int dev = ctn_current_device();
  if (!attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_wgrad_umma<NPASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr_done[dev] = true;
  }
  k_wgrad_umma<NPASS><<<grid, WG_THREADS, smem, st>>>(g);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  return CTN_OK;
}

}  // namespace

// rows [0, split_row) of the (M, K) result go to dWa, the rest to dWb (pass split_row = M and dWb = nullptr for one tensor)
int ctn_wgrad_umma(const float* dy, size_t dy_bs, const float* x, size_t x_bs, float* dWa, float* dWb, int split_row, int M,
                   int K, int B, int frames, int pitch, int math, cudaStream_t st) {
  if (!dy || !x || !dWa || M <= 0 || K <= 0 || B <= 0 || frames <= 0) return CTN_EINVAL;
  if (pitch % 128 != 0 || (dy_bs % 4) != 0 || (x_bs % 4) != 0) return CTN_EALIGN;
  if ((((uintptr_t)dy) | ((uintptr_t)x)) & 15) return CTN_EALIGN;
  WgArgs g;
  memset(&g, 0, sizeof(g));
  g.dy = dy; g.dy_bs = dy_bs; g.x = x; g.x_bs = x_bs; g.dWa = dWa; g.dWb = dWb; g.split_row = dWb ? split_row : M;
  g.M = M; g.K = K; g.B = B; g.frames = frames; g.pitch = pitch;
  g.n_tile = K >= 256 ? 256 : ((K + 31) / 32) * 32;  // the producers stage X in groups of 32 rows
  g.tiles_n = (K + g.n_tile - 1) / g.n_tile;
  g.tiles = ((M + 127) / 128) * g.tiles_n;
  g.chunks = (frames + WG_KT - 1) / WG_KT;
  const long long total = (long long)B * g.chunks;
  long long splits = ctn_num_sms() / g.tiles;
  if (splits < 1) splits = 1;
  if (splits > total) splits = total;
  g.steps_per_split = (int)((total + splits - 1) / splits);
  splits = (total + g.steps_per_split - 1) / g.steps_per_split;
  const int nprec = math == CTN_MATH_TF32 ? 1 : 2;  // F16X3 forwards use the 3xTF32 weight-gradient kernel
  g.stage_bytes = (uint32_t)nprec * (WG_A_BYTES + (uint32_t)g.n_tile * 128u);
  int stages = (int)((227 * 1024 - WG_HEADER - 1024) / g.stage_bytes);
  if (stages > WG_MAX_STAGES) stages = WG_MAX_STAGES;
  if (stages < 2) return CTN_EUNSUPPORTED;
  g.stages = stages;
  g.idesc = ptx::make_idesc_tf32(128, g.n_tile, /*A K-major*/ 0, /*B K-major*/ 0);
  g.tmem_cols = 32;
  while ((int)g.tmem_cols < g.n_tile) g.tmem_cols <<= 1;
  const size_t smem = WG_HEADER + 1024 + (size_t)stages * g.stage_bytes;
  const int grid = g.tiles * (int)splits;
  return nprec == 2 ? launch_wg<3>(g, smem, grid, st) : launch_wg<1>(g, smem, grid, st);
}
