// extern "C" entry points + host-side orchestration of the Conv-TasNet forward (see include/ctn_b200.h).
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "ctn_internal.h"

thread_local int g_ctn_launches = 0;
thread_local long long g_ctn_total_launches = 0;
thread_local int g_ctn_depth = 0;
thread_local int g_ctn_last_launches = 0;

// ---- stage profiler ---------------------------------------------------------------------------------------
struct ProfRec { int stage; cudaEvent_t e0, e1; int launches0, launches; };
static thread_local bool g_prof_on = false;
static thread_local std::vector<ProfRec> g_prof_recs;
static thread_local std::vector<cudaEvent_t> g_prof_pool;
static thread_local int g_prof_depth = 0;
static cudaEvent_t prof_event() {
  cudaEvent_t e;
  if (!g_prof_pool.empty()) { e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEventCreate(&e);
  return e;
}
void ctn_prof_begin(int stage, cudaStream_t st) {
  if (!g_prof_on || g_prof_depth++ > 0) return;
  ProfRec r;
  r.stage = stage; r.e0 = prof_event(); r.e1 = prof_event(); r.launches0 = g_ctn_launches; r.launches = 0;
  cudaEventRecord(r.e0, st);
  g_prof_recs.push_back(r);
}
void ctn_prof_end(int stage, cudaStream_t st) {
  if (!g_prof_on || --g_prof_depth > 0) return;
  ProfRec& r = g_prof_recs.back();
  r.launches = g_ctn_launches - r.launches0;
  cudaEventRecord(r.e1, st);
}
extern "C" int ctn_profile_enable(int enable) { g_prof_on = enable != 0; g_prof_depth = 0; return CTN_OK; }
extern "C" int ctn_profile_read(double* ms, int* launches) {
  if (!ms || !launches) return CTN_EINVAL;
  for (ProfRec& r : g_prof_recs) {
    cudaError_t e = cudaEventSynchronize(r.e1);
    if (e != cudaSuccess) return (int)e;
    float t = 0.f;
    e = cudaEventElapsedTime(&t, r.e0, r.e1);
    if (e != cudaSuccess) return (int)e;
    ms[r.stage] += (double)t;
    launches[r.stage] += r.launches;
    g_prof_pool.push_back(r.e0);
    g_prof_pool.push_back(r.e1);
  }
  g_prof_recs.clear();
  return CTN_OK;
}

extern "C" int ctn_version(void) { return CTN_VERSION; }
extern "C" int ctn_last_launch_count(void) { return g_ctn_last_launches; }
extern "C" long long ctn_total_launch_count(void) { return g_ctn_total_launches; }

extern "C" const char* ctn_strerror(int s) {
  switch (s) {
    case CTN_OK: return "ok";
    case CTN_EINVAL: return "invalid argument (shape / null pointer)";
    case CTN_EUNSUPPORTED: return "configuration outside the kernel envelope";
    case CTN_EALIGN: return "pointer or pitch alignment";
    case CTN_EWORKSPACE: return "workspace too small";
    case CTN_ENOTBUILT: return "kernel family not built into this library";
    default: return s > 0 ? cudaGetErrorString((cudaError_t)s) : "unknown ctn error";
  }
}

extern "C" int ctn_frames(int T, int kernel_size, int stride, int* pad_left, int* pad_right) {
  if (T <= 0 || kernel_size <= 0 || stride <= 0 || kernel_size % stride != 0) return CTN_EINVAL;
  // src/models/conv_tasnet.py:145-147
  int r = (T - kernel_size) % stride;
  if (r < 0) r += stride;  // python modulo
  const int padding = (stride - r) % stride;
  const int pl = padding / 2, pr = padding - pl;
  if (pad_left) *pad_left = pl;
  if (pad_right) *pad_right = pr;
  const int Tp = T + padding;
  if (Tp < kernel_size) return CTN_EINVAL;
  return (Tp - kernel_size) / stride + 1;
}

extern "C" int ctn_pitch(int frames) { return frames <= 0 ? CTN_EINVAL : ctn_round_up(frames, CTN_TILE_T); }

// ------------------------------------------------------------------------------------------------
// workspace carving
// ------------------------------------------------------------------------------------------------
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

struct TcnWs {
  double* stats;  // [2*RX][B][2]
  std::vector<FoldedConv> folds;  // per block, (Bc+Sc) rows
  std::vector<float*> wimg1, wimg2;  // per block: tcgen05 weight images of the two pointwise convs (math != fp32)
  std::vector<float*> rblk;          // per block: raw [out;skip] contraction output r_i (B, Bc+Sc, pitch), kept for the
                                     // deferred skip reduction (the skip accumulator is written once, at the end)
  float *x, *skip, *h, *u, *outraw;
  void* causal_ws;  // causal (cLN) models: scratch of the un-fused pipeline (ctn_causal.cu)
  float* xalt;  // second residual-stream buffer (tcgen05 modes ping-pong x between blocks: the update is fused into pw1)
  // fp16-piece mode: activation envelope (ctn_act_scales)
  std::vector<float*> dwp;  // per block: packed depthwise parameters [ceil16(H)][8]
  float* scales;            // [2*RX + 1] power-of-two operand scales (+ 3*RX floats of scratch)
  float* x0_bound;          // [x0_n] candidates bounding |x_0|: the head's per-row bounds, or the measured max |x| (ctn_tcn_fwd)
  int x0_n;
  const float* mask_slope;  // separator.prelu (nullable)
  size_t stats_bytes;
};

static int check_tcn_cfg(const ctn_config_t* c) {
  if (!c) return CTN_EINVAL;
  if (c->bottleneck <= 0 || c->hidden <= 0 || c->skip <= 0 || c->sep_kernel <= 0 || c->num_blocks <= 0 || c->num_layers <= 0)
    return CTN_EINVAL;
  if (c->num_layers > 20 || c->num_blocks * c->num_layers > CTN_MAX_BLOCKS) return CTN_EUNSUPPORTED;
  if (c->math != CTN_MATH_FP32 && c->math != CTN_MATH_TF32X3 && c->math != CTN_MATH_TF32 && c->math != CTN_MATH_F16X3) return CTN_EINVAL;
  return CTN_OK;
}

static void carve_tcn(Carver& cv, const ctn_config_t* c, int B, int pitch, TcnWs* ws) {
  const int RX = c->num_blocks * c->num_layers;
  const int Mt = c->bottleneck + c->skip;
  ws->stats_bytes = sizeof(double) * 2 * RX * B * 2;
  ws->stats = cv.take<double>((size_t)2 * RX * B * 2);
  ws->folds.resize(RX);
  ws->wimg1.assign(RX, nullptr);
  ws->wimg2.assign(RX, nullptr);
  for (int i = 0; i < RX; ++i) {
    ws->folds[i].Wf = cv.take<float>((size_t)Mt * c->hidden);
    ws->folds[i].v1 = cv.take<float>(Mt);
    ws->folds[i].v2 = cv.take<float>(Mt);
    ws->folds[i].vb = cv.take<float>(Mt);
    if (c->math != CTN_MATH_FP32) {
      ws->wimg1[i] = cv.take<float>(ctn_umma_wimg_bytes(c->hidden, c->bottleneck, c->math) / sizeof(float));
      ws->wimg2[i] = cv.take<float>(ctn_umma_wimg_bytes(Mt, c->hidden, c->math) / sizeof(float));
    }
  }
  ws->dwp.assign(RX, nullptr);
  for (int i = 0; i < RX; ++i) ws->dwp[i] = cv.take<float>((size_t)ctn_round_up(c->hidden, 16) * 8);
  ws->scales = cv.take<float>((size_t)5 * RX + 8);
  ws->x0_bound = cv.take<float>(64);  // ctn_tcn_fwd: measured max |x|; the model path points x0_bound at the head's row bounds
  ws->x0_n = 1;
  ws->mask_slope = nullptr;
  const size_t bp = (size_t)B * pitch;
  ws->x = cv.take<float>(bp * c->bottleneck);
  ws->xalt = cv.take<float>(bp * c->bottleneck);
  ws->skip = cv.take<float>(bp * c->skip);
  ws->h = cv.take<float>(bp * c->hidden);
  ws->u = cv.take<float>(bp * c->hidden);
  ws->outraw = nullptr;
  ws->rblk.assign(RX, nullptr);
  ws->causal_ws = nullptr;
  if (c->causal) {
    ws->causal_ws = cv.take<char>(ctn_causal_ws_bytes(c, B, pitch));
  } else {
    for (int i = 0; i < RX; ++i) ws->rblk[i] = cv.take<float>(bp * Mt);
  }
}

static int pw_dispatch(const PwArgs& a, int pro, int epi, int math, cudaStream_t st) {
  if (math == CTN_MATH_FP32) return ctn_pw_simt(a, pro, epi, st);
  if (math == CTN_MATH_F16X3 && ctn_pw_tma_supported(a, pro, epi)) return ctn_pw_tma(a, pro, epi, st);
  return ctn_pw_umma(a, pro, epi, math, st);
}

// TCN over ws->x (padded layout) -> ws->skip.  stats region must be zeroed by the caller.
// dil (nullable): explicit dilation per block (ctn_tcn_blocks_fwd); default 2^layer (dilated=True, tdcn.py:52-54).
// x_final (nullable): receives a pointer to the residual stream AFTER the last block (x_n), updated in the workspace.
// hooks (nullable): TRAINING forward through the fused kernels -- block i reads its input from x_keep[i] (x_keep[0] = the head's
// output, filled by the caller) and leaves x_{i+1} in x_keep[i+1]; pw1 stores the PRE-activation W1 x + b1 in hpre[i], the fused
// depthwise producer applies PReLU on load and stores its own pre-activation in upre[i] (what ctn_convtasnet_bwd consumes).
static int run_tcn(const ctn_config_t* c, const ctn_block_params_t* blocks, TcnWs* ws, int B, int frames, int pitch,
                   cudaStream_t st, const int* dil = nullptr, float** x_final = nullptr, const TcnTrainHooks* hooks = nullptr) {
  const int R = c->num_blocks, X = c->num_layers, Bc = c->bottleneck, H = c->hidden, Sc = c->skip;
  if (c->causal)  // cLN: cumulative statistics -> un-fused pipeline in the reference's operation order
    return ctn_causal_tcn(c, blocks, ws->x, ws->skip, ws->h, ws->u, B, frames, pitch, ws->causal_ws, st);
  // weight preparation for all blocks: gLN2 folding, then (tcgen05 modes) the swizzled hi/lo operand images
  {
    StageTimer tm(CTN_ST_PREP, st);
    std::vector<FoldJob> fj;
    std::vector<WimgJob> wj;
    const float Rh = sqrtf((float)H * (float)frames) * 1.0001f;  // >= max |normalised value| of a gLN group of H*frames elements
    ScaleJobs* sj = new ScaleJobs;
    memset(sj, 0, sizeof(*sj));
    for (int i = 0; i < R * X; ++i) {
      const ctn_block_params_t& p = blocks[i];
      const bool has_out = p.out_w != nullptr;
      const FoldedConv& f = ws->folds[i];
      if (has_out) fj.push_back(FoldJob{p.out_w, p.out_b, p.norm2_g, p.norm2_b, f.Wf, f.v1, f.v2, Bc, H, 0, f.vb, Rh});
      fj.push_back(FoldJob{p.skip_w, p.skip_b, p.norm2_g, p.norm2_b, f.Wf, f.v1, f.v2, Sc, H, has_out ? Bc : 0, f.vb, Rh});
      sj->j[i] = ScaleJob{f.vb, p.norm1_g, p.norm1_b, p.dw_w, p.dw_b, p.prelu2, ws->dwp[i], has_out ? 1 : 0};
      if (c->math != CTN_MATH_FP32) {
        wj.push_back(WimgJob{p.bottleneck_w, ws->wimg1[i], H, Bc});
        wj.push_back(WimgJob{f.Wf, ws->wimg2[i], has_out ? Bc + Sc : Sc, H});
      }
    }
    int rc = ctn_fold_batch(fj.data(), (int)fj.size(), st);
    if (rc == CTN_OK && !wj.empty()) rc = ctn_umma_build_wimg_batch(wj.data(), (int)wj.size(), c->math, st);
    if (rc == CTN_OK && c->math == CTN_MATH_F16X3) {
      sj->n = R * X; sj->Bc = Bc; sj->Sc = Sc; sj->H = H; sj->P = c->sep_kernel; sj->R = Rh;
      sj->x0_bound = ws->x0_bound; sj->x0_n = ws->x0_n; sj->mask_slope = ws->mask_slope; sj->scales = ws->scales;
      rc = ctn_act_scales(*sj, st);
    }
    delete sj;
    CTN_TRY(rc);
  }
  const bool scaled = c->math == CTN_MATH_F16X3;
  for (int r = 0; r < R; ++r) {
    for (int l = 0; l < X; ++l) {
      const int i = r * X + l;
      const ctn_block_params_t& p = blocks[i];
      const bool has_out = p.out_w != nullptr;
      if (!has_out && !(r == R - 1 && l == X - 1)) return CTN_EINVAL;
      const int dilation = dil ? dil[i] : (1 << l);  // dilated=True (tdcn.py:52-54)
      double* st1 = ws->stats + (size_t)(2 * i) * B * 2;
      double* st2 = ws->stats + (size_t)(2 * i + 1) * B * 2;
      // K_A: h = PReLU(W1 x + b1), stats1
      PwArgs a;
      memset(&a, 0, sizeof(a));
      // tcgen05 modes: the residual stream ping-pongs between ws->x and ws->xalt; block i >= 1 applies block i-1's
      // update x += rstd2*r[:Bc] + c inside its own producer (PRO_RES) -- no separate finishing pass over x
      const bool fuse_res = c->math != CTN_MATH_FP32;
      float* xbuf[2] = {ws->x, ws->xalt};
      // training forward: per-block buffers; x_i is read from x_keep[i] (written by block i-1 below), kept for the backward
      if (hooks && !fuse_res) return CTN_EUNSUPPORTED;
      float* const hbuf = hooks ? hooks->hpre[i] : ws->h;
      a.A = fuse_res ? xbuf[(i + 1) & 1] : xbuf[0];
      if (fuse_res && i == 0) a.A = hooks ? hooks->x_keep[0] : xbuf[0];
      a.W = p.bottleneck_w; a.D = hbuf; a.B = B; a.M = H; a.K = Bc; a.frames = frames; a.pitch = pitch;
      a.store_pre = hooks ? 1 : 0;
      a.bias = p.bottleneck_b; a.slope = p.prelu1; a.stats_out = st1; a.wimg = ws->wimg1[i];
      if (scaled) a.act_scale = ws->scales + 2 * i;
      int pro1 = PRO_NONE;
      if (fuse_res && i > 0) {
        // x_{i} = x_{i-1} + deferred gLN2 of block i-1;  x_{i-1} lives in xbuf[(i-1)&1], x_i goes to xbuf[i&1]
        pro1 = PRO_RES;
        a.A = hooks ? hooks->x_keep[i - 1] : xbuf[(i - 1) & 1];
        a.res_r = ws->rblk[i - 1]; a.res_Mt = Bc + Sc;  // block i-1 always has the out head (only the last block lacks it)
        a.res_v1 = ws->folds[i - 1].v1; a.res_v2 = ws->folds[i - 1].v2;
        a.res_stats = ws->stats + (size_t)(2 * (i - 1) + 1) * B * 2; a.res_n = (double)H * (double)frames; a.res_eps = c->eps_tcn;
        a.res_x_out = hooks ? hooks->x_keep[i] : xbuf[i & 1];
      }
      if (hooks && !(c->math == CTN_MATH_F16X3 && ctn_pw_tma_supported(a, pro1, EPI_H))) return CTN_EUNSUPPORTED;
      { StageTimer tm(CTN_ST_PW1, st); CTN_TRY(pw_dispatch(a, pro1, EPI_H, c->math, st)); }
      const int Mt = has_out ? Bc + Sc : Sc;
      float* rb = ws->rblk[i];
      const int pad_left = c->causal ? (c->sep_kernel - 1) * dilation : ((c->sep_kernel - 1) * dilation) / 2;
      // fused depthwise producer: 3 taps at dilation 1, 2 or a multiple of 4 (128-bit aligned tap loads); anything else runs the
      // stand-alone depthwise stage
      const bool dw_fusable = c->sep_kernel == 3 && (dilation == 1 || dilation == 2 || dilation % 4 == 0);
      if (c->math != CTN_MATH_FP32 && dw_fusable) {
        // K_BC fused (tcgen05): the producer warps compute u = PReLU(dwconv(gLN1(h))) (+stats2) on the fly and feed
        // it straight to the tensor core; u never touches HBM.  r = [Wo;Ws] diag(gamma2) u
        StageTimer tm(CTN_ST_PW2, st);
        memset(&a, 0, sizeof(a));
        a.A = hbuf; a.W = ws->folds[i].Wf; a.D = rb; a.B = B; a.M = Mt; a.K = H; a.frames = frames; a.pitch = pitch;
        a.wimg = ws->wimg2[i];
        a.pro_slope = p.prelu2; a.dw_norm_g = p.norm1_g; a.dw_norm_b = p.norm1_b; a.dw_w = p.dw_w; a.dw_b = p.dw_b;
        a.dw_stats_in = st1; a.dw_stats_out = st2; a.dw_dilation = dilation; a.dw_pad_left = pad_left; a.dw_eps = c->eps_tcn;
        if (scaled) { a.act_scale = ws->scales + 2 * i + 1; a.dw_params = ws->dwp[i]; }
        if (hooks) {
          a.dw_in_slope = p.prelu1; a.dw_u_pre_out = hooks->upre[i];
          if (!(c->math == CTN_MATH_F16X3 && ctn_pw_tma_supported(a, PRO_DW, EPI_RAW))) return CTN_EUNSUPPORTED;
        }
        CTN_TRY(pw_dispatch(a, PRO_DW, EPI_RAW, c->math, st));
      } else {
        if (hooks) return CTN_EUNSUPPORTED;
        // K_B: u = PReLU(dwconv(gLN1(h))), stats2
        { StageTimer tm(CTN_ST_DW, st);
          CTN_TRY(ctn_dw_fwd(hbuf, ws->u, p.norm1_g, p.norm1_b, p.dw_w, p.dw_b, p.prelu2, st1, st2, B, H, frames, pitch,
                             c->sep_kernel, dilation, c->causal, c->eps_tcn, st)); }
        // K_C: r = [Wo;Ws] diag(gamma2) u
        memset(&a, 0, sizeof(a));
        a.A = ws->u; a.W = ws->folds[i].Wf; a.D = rb; a.B = B; a.M = Mt; a.K = H; a.frames = frames; a.pitch = pitch;
        a.wimg = ws->wimg2[i];
        if (scaled) a.act_scale = ws->scales + 2 * i + 1;
        { StageTimer tm(CTN_ST_PW2, st); CTN_TRY(pw_dispatch(a, PRO_NONE, EPI_RAW, c->math, st)); }
      }
      // K_F: residual update with the deferred gLN2 (x += rstd2*r[:Bc] + c); the skip rows are reduced once at the end
      if (has_out && c->math == CTN_MATH_FP32) {
        StageTimer tm(CTN_ST_FIN, st);
        CTN_TRY(ctn_finish_fwd(rb, ws->folds[i], st2, (double)H * (double)frames, c->eps_tcn, xbuf[0], ws->skip, B, Bc,
                               Sc, 1, 2 /* x rows only */, frames, pitch, st));
      }
    }
  }
  {
    StageTimer tm(CTN_ST_FIN, st);
    SkipJobs sj;
    sj.n = R * X;
    for (int i = 0; i < R * X; ++i) {
      const bool has_out = blocks[i].out_w != nullptr;
      sj.j[i] = SkipJob{ws->rblk[i], ws->folds[i].v1, ws->folds[i].v2, ws->stats + (size_t)(2 * i + 1) * B * 2, has_out ? Bc : 0,
                        has_out ? Bc + Sc : Sc};
    }
    CTN_TRY(ctn_skip_reduce(sj, (double)H * (double)frames, c->eps_tcn, ws->skip, B, Sc, frames, pitch, st));
  }
  if (x_final) {
    const int n = R * X;
    float* xbuf[2] = {ws->x, ws->xalt};
    float* xl = (c->math != CTN_MATH_FP32) ? xbuf[(n - 1) & 1] : ws->x;  // x_{n-1} (tcgen05 modes defer every update to the next block)
    if (c->math != CTN_MATH_FP32 && blocks[n - 1].out_w)
      CTN_TRY(ctn_finish_fwd(ws->rblk[n - 1], ws->folds[n - 1], ws->stats + (size_t)(2 * (n - 1) + 1) * B * 2, (double)H * (double)frames,
                             c->eps_tcn, xl, ws->skip, B, Bc, Sc, 1, 2 /* x rows only */, frames, pitch, st));
    *x_final = xl;
  }
  return CTN_OK;
}

// ---- training forward through the fused kernels (called by ctn_convtasnet_fwd_train, ctn_train.cu) ----------------------------
// The training workspace carries its own copy of the small per-forward state of the TCN (folds, weight images, depthwise
// parameter packs, operand scales) and one raw [out;skip] tensor per block; x / h_pre / u_pre live in the caller's per-block
// buffers, the statistics in the caller's array (same [2*RX][B][2] layout the backward reads).
static void carve_tcn_train(Carver& cv, const ctn_config_t* c, int B, int pitch, TcnWs* ws) {
  const int RX = c->num_blocks * c->num_layers;
  const int Mt = c->bottleneck + c->skip;
  ws->stats = nullptr; ws->stats_bytes = 0;
  ws->folds.resize(RX);
  ws->wimg1.assign(RX, nullptr);
  ws->wimg2.assign(RX, nullptr);
  ws->dwp.assign(RX, nullptr);
  ws->rblk.assign(RX, nullptr);
  for (int i = 0; i < RX; ++i) {
    ws->folds[i].Wf = cv.take<float>((size_t)Mt * c->hidden);
    ws->folds[i].v1 = cv.take<float>(Mt);
    ws->folds[i].v2 = cv.take<float>(Mt);
    ws->folds[i].vb = cv.take<float>(Mt);
    ws->wimg1[i] = cv.take<float>(ctn_umma_wimg_bytes(c->hidden, c->bottleneck, c->math) / sizeof(float));
    ws->wimg2[i] = cv.take<float>(ctn_umma_wimg_bytes(Mt, c->hidden, c->math) / sizeof(float));
    ws->dwp[i] = cv.take<float>((size_t)ctn_round_up(c->hidden, 16) * 8);
    ws->rblk[i] = cv.take<float>((size_t)B * pitch * Mt);
  }
  ws->scales = cv.take<float>((size_t)5 * RX + 8);
  ws->x0_bound = cv.take<float>(64);
  ws->x0_n = 1;
  ws->mask_slope = nullptr;
  ws->x = ws->xalt = ws->skip = ws->h = ws->u = ws->outraw = nullptr;
  ws->causal_ws = nullptr;
}
size_t ctn_tcn_train_ws_bytes(const ctn_config_t* c, int B, int pitch) {
  Carver cv(nullptr);
  TcnWs ws;
  carve_tcn_train(cv, c, B, pitch, &ws);
  return cv.off + 512;
}
int ctn_tcn_train_fwd(const ctn_config_t* c, const ctn_block_params_t* blocks, void* mem, size_t mem_bytes, const TcnTrainHooks* hooks,
                      double* stats, float* skip, const float* x0_bound, int x0_n, const float* mask_slope, const float** mask_scale,
                      int B, int frames, int pitch, cudaStream_t st) {
  if (!c || !blocks || !mem || !hooks || !stats || !skip || (((uintptr_t)mem) & 255)) return CTN_EINVAL;
  if (c->math != CTN_MATH_F16X3 || c->causal || c->sep_kernel != 3) return CTN_EUNSUPPORTED;
  if (mem_bytes < ctn_tcn_train_ws_bytes(c, B, pitch)) return CTN_EWORKSPACE;
  Carver cv(mem);
  TcnWs ws;
  carve_tcn_train(cv, c, B, pitch, &ws);
  ws.stats = stats;
  ws.skip = skip;
  ws.x0_bound = const_cast<float*>(x0_bound);
  ws.x0_n = x0_n;
  ws.mask_slope = mask_slope;
  CTN_TRY(run_tcn(c, blocks, &ws, B, frames, pitch, st, nullptr, nullptr, hooks));
  if (mask_scale) *mask_scale = ws.scales + 2 * c->num_blocks * c->num_layers;
  return CTN_OK;
}

extern "C" int ctn_tcn_workspace_bytes(const ctn_config_t* cfg, int batch, int frames, size_t* bytes) {
  CTN_TRY(check_tcn_cfg(cfg));
  if (batch <= 0 || frames <= 0 || !bytes) return CTN_EINVAL;
  Carver cv(nullptr);
  TcnWs ws;
  carve_tcn(cv, cfg, batch, ctn_pitch(frames), &ws);
  *bytes = cv.off + 256;
  return CTN_OK;
}

extern "C" int ctn_tcn_fwd(const ctn_config_t* cfg, const ctn_block_params_t* blocks, const float* x, float* skip_out, int B,
                           int frames, void* workspace, size_t workspace_bytes, ctn_stream_t stream) {
  LaunchScope scope(x);
  CTN_TRY(check_tcn_cfg(cfg));
  if (!blocks || !x || !skip_out || !workspace || B <= 0 || frames <= 0) return CTN_EINVAL;
  if (((uintptr_t)workspace) & 255) return CTN_EALIGN;
  size_t need = 0;
  CTN_TRY(ctn_tcn_workspace_bytes(cfg, B, frames, &need));
  if (workspace_bytes < need) return CTN_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int pitch = ctn_pitch(frames);
  Carver cv(workspace);
  TcnWs ws;
  carve_tcn(cv, cfg, B, pitch, &ws);
  cudaError_t e = cudaMemsetAsync(ws.stats, 0, ws.stats_bytes, st);
  if (e != cudaSuccess) return (int)e;
  CTN_TRY(ctn_copy_to_pitch(x, ws.x, B * cfg->bottleneck, frames, pitch, st));
  if (cfg->math == CTN_MATH_F16X3 && !cfg->causal) {  // stand-alone TCN: |x_0| is whatever the caller passes -- measure it
    e = cudaMemsetAsync(ws.x0_bound, 0, sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
    CTN_TRY(ctn_absmax_pitch(ws.x, B * cfg->bottleneck, frames, pitch, ws.x0_bound, st));
  }
  CTN_TRY(run_tcn(cfg, blocks, &ws, B, frames, pitch, st));
  CTN_TRY(ctn_copy_from_pitch(ws.skip, skip_out, B * cfg->skip, frames, pitch, st));
  return CTN_OK;
}

// A run of residual blocks with explicit dilations, returning BOTH heads: ResidualBlock1d.forward (tdcn.py:107-147, n = 1) and
// TimeDilatedConvBlock1d.forward (tdcn.py:65-75): x (B,Bc,frames) -> x_out (nullable; the residual stream after the last block,
// which must have the output head) and skip_out (B,Sc,frames) = sum of the blocks' skip heads.  cfg as for ctn_tcn_fwd
// (num_blocks * num_layers is ignored; n_blocks counts).
extern "C" int ctn_tcn_blocks_fwd(const ctn_config_t* cfg, const ctn_block_params_t* blocks, int n_blocks, const int* dilations,
                                  const float* x, float* x_out, float* skip_out, int B, int frames, void* workspace,
                                  size_t workspace_bytes, ctn_stream_t stream) {
  LaunchScope scope(x);
  if (!cfg || !blocks || !dilations || n_blocks <= 0 || n_blocks > CTN_MAX_BLOCKS || !x || !skip_out || !workspace || B <= 0 || frames <= 0)
    return CTN_EINVAL;
  ctn_config_t c = *cfg;
  c.num_blocks = 1;
  c.num_layers = n_blocks;
  if (c.bottleneck <= 0 || c.hidden <= 0 || c.skip <= 0 || c.sep_kernel <= 0) return CTN_EINVAL;
  if (c.causal) return CTN_EUNSUPPORTED;  // the causal pipeline takes its dilations from the layer index
  for (int i = 0; i < n_blocks; ++i) {
    if (dilations[i] < 1) return CTN_EINVAL;
    if (!blocks[i].out_w && i != n_blocks - 1) return CTN_EINVAL;
  }
  if (x_out && !blocks[n_blocks - 1].out_w) return CTN_EINVAL;
  if (((uintptr_t)workspace) & 255) return CTN_EALIGN;
  const int pitch = ctn_pitch(frames);
  Carver cv0(nullptr);
  TcnWs ws;
  carve_tcn(cv0, &c, B, pitch, &ws);
  if (workspace_bytes < cv0.off + 256) return CTN_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(workspace);
  carve_tcn(cv, &c, B, pitch, &ws);
  cudaError_t e = cudaMemsetAsync(ws.stats, 0, ws.stats_bytes, st);
  if (e != cudaSuccess) return (int)e;
  CTN_TRY(ctn_copy_to_pitch(x, ws.x, B * c.bottleneck, frames, pitch, st));
  if (c.math == CTN_MATH_F16X3) {
    e = cudaMemsetAsync(ws.x0_bound, 0, sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
    CTN_TRY(ctn_absmax_pitch(ws.x, B * c.bottleneck, frames, pitch, ws.x0_bound, st));
  }
  float* xf = nullptr;
  CTN_TRY(run_tcn(&c, blocks, &ws, B, frames, pitch, st, dilations, x_out ? &xf : nullptr));
  if (x_out) CTN_TRY(ctn_copy_from_pitch(xf, x_out, B * c.bottleneck, frames, pitch, st));
  CTN_TRY(ctn_copy_from_pitch(ws.skip, skip_out, B * c.skip, frames, pitch, st));
  return CTN_OK;
}

// ------------------------------------------------------------------------------------------------
// full model
// ------------------------------------------------------------------------------------------------
struct ModelWs {
  double* stats0;  // [B][2]
  FoldedConv head; // (Bc, N)
  float* w;        // (B, N, pitch)
  float* what;     // (B, S*N, pitch)
  float *wimg_head, *wimg_mask;
  TcnWs tcn;
};

static int check_model_cfg(const ctn_config_t* c) {
  CTN_TRY(check_tcn_cfg(c));
  if (c->n_basis <= 0 || c->kernel_size <= 0 || c->stride <= 0 || c->n_sources <= 0) return CTN_EINVAL;
  if (c->kernel_size % c->stride != 0) return CTN_EINVAL;
  if (c->mask_softmax && c->mask_softmax != 1) return CTN_EINVAL;
  if (c->in_channels < 0 || c->in_channels > 64) return CTN_EINVAL;
  return CTN_OK;
}

static void carve_model(Carver& cv, const ctn_config_t* c, int B, int pitch, ModelWs* ws) {
  ws->stats0 = cv.take<double>((size_t)B * 2);
  ws->head.Wf = cv.take<float>((size_t)c->bottleneck * c->n_basis);
  ws->head.v1 = cv.take<float>(c->bottleneck);
  ws->head.v2 = cv.take<float>(c->bottleneck);
  ws->head.vb = cv.take<float>(c->bottleneck);
  ws->wimg_head = ws->wimg_mask = nullptr;
  if (c->math != CTN_MATH_FP32) {
    ws->wimg_head = cv.take<float>(ctn_umma_wimg_bytes(c->bottleneck, c->n_basis, c->math) / sizeof(float));
    ws->wimg_mask = cv.take<float>(ctn_umma_wimg_bytes(c->n_sources * c->n_basis, c->skip, c->math) / sizeof(float));
  }
  const size_t bp = (size_t)B * pitch;
  ws->w = cv.take<float>(bp * c->n_basis);
  ws->what = cv.take<float>(bp * c->n_basis * c->n_sources);
  carve_tcn(cv, c, B, pitch, &ws->tcn);
}

extern "C" int ctn_workspace_bytes(const ctn_config_t* cfg, int batch, int T, size_t* bytes) {
  CTN_TRY(check_model_cfg(cfg));
  if (batch <= 0 || !bytes) return CTN_EINVAL;
  const int frames = ctn_frames(T, cfg->kernel_size, cfg->stride, nullptr, nullptr);
  if (frames <= 0) return CTN_EINVAL;
  Carver cv(nullptr);
  ModelWs ws;
  carve_model(cv, cfg, batch, ctn_pitch(frames), &ws);
  *bytes = cv.off + 256;
  return CTN_OK;
}

// separator on ws->w (+ stats0 already accumulated) -> ws->what (= w*mask) and optionally the raw mask
// dec (nullable): when the fused mask + decoder epilogue applies (fp16-piece mode, kernel 16 / stride 8, no mask / latent output
// wanted) the estimates are written straight to dec->out and dec->fused is set; w_hat is then never materialised
struct DecFuse { float* out; int crop_left, T_out; bool fused; };
static int run_separator(const ctn_config_t* c, const ctn_params_t* p, ModelWs* ws, int B, int frames, int pitch,
                         float* mask_out, cudaStream_t st, DecFuse* dec = nullptr) {
  const int N = c->n_basis, Bc = c->bottleneck, Sc = c->skip, S = c->n_sources;
  if (c->causal) {
    // cLN0 -> bottleneck 1x1; ws->what is free until the mask kernel writes it: use it as the (B, N, pitch) scratch
    CTN_TRY(ctn_causal_head(c, p, ws->w, ws->what, ws->tcn.x, B, frames, pitch, ws->tcn.causal_ws, st));
    if (c->math != CTN_MATH_FP32) {
      StageTimer tm(CTN_ST_PREP, st);
      CTN_TRY(ctn_umma_build_wimg(p->mask_w, S * N, Sc, c->math == CTN_MATH_F16X3 ? CTN_MATH_TF32X3 : c->math, ws->wimg_mask, st));
    }
  } else {
    // head: gLN0 folded into the bottleneck 1x1 (conv_tasnet.py:370-371).  Its operand is the un-normalised encoder output
    // (any input scale), so the fp16-piece mode falls back to the tf32 pieces here (0.14 ms of the step).
    const int head_math = c->math == CTN_MATH_F16X3 ? CTN_MATH_TF32X3 : c->math;
    { StageTimer tm(CTN_ST_PREP, st);
      CTN_TRY(ctn_fold_conv(p->bn_w, p->bn_b, p->norm0_g, p->norm0_b, Bc, N, ws->head, 0, st, sqrtf((float)N * (float)frames) * 1.0001f));
      if (c->math != CTN_MATH_FP32) {
        CTN_TRY(ctn_umma_build_wimg(ws->head.Wf, Bc, N, head_math, ws->wimg_head, st));
        CTN_TRY(ctn_umma_build_wimg(p->mask_w, S * N, Sc, c->math, ws->wimg_mask, st));
      }
    }
    PwArgs a;
    memset(&a, 0, sizeof(a));
    a.A = ws->w; a.W = ws->head.Wf; a.D = ws->tcn.x; a.B = B; a.M = Bc; a.K = N; a.frames = frames; a.pitch = pitch;
    a.v1 = ws->head.v1; a.v2 = ws->head.v2; a.stats_in = ws->stats0; a.n_in = (double)N * (double)frames; a.eps = c->eps;
    a.wimg = ws->wimg_head;
    { StageTimer tm(CTN_ST_HEAD, st); CTN_TRY(pw_dispatch(a, PRO_NONE, EPI_HEAD, head_math, st)); }
  }
  // TCN (conv_tasnet.py:372).  fp16-piece mode: |x_0| <= max_n of the head's row bounds; the mask operand is PReLU(skip sum)
  ws->tcn.x0_bound = ws->head.vb; ws->tcn.x0_n = Bc; ws->tcn.mask_slope = p->prelu_out;
  CTN_TRY(run_tcn(c, p->blocks, &ws->tcn, B, frames, pitch, st));
  // tail: PReLU -> mask 1x1 -> sigmoid -> * w  (conv_tasnet.py:373-376, 159-160)
  PwArgs a;
  memset(&a, 0, sizeof(a));
  a.A = ws->tcn.skip; a.W = p->mask_w; a.D = ws->what; a.B = B; a.M = S * N; a.K = Sc; a.frames = frames; a.pitch = pitch;
  a.pro_slope = p->prelu_out; a.bias = p->mask_b; a.wenc = ws->w; a.Nb = N; a.mask_out = mask_out; a.wimg = ws->wimg_mask;
  if (c->math == CTN_MATH_F16X3 && !c->causal) a.act_scale = ws->tcn.scales + 2 * c->num_blocks * c->num_layers;
  // causal models: no operand scales (un-fused pipeline) -> the mask contraction stays on the tf32 pieces
  const int mask_math = (c->causal && c->math == CTN_MATH_F16X3) ? CTN_MATH_TF32X3 : c->math;
  if (c->mask_softmax) {
    // nn.Softmax(dim=1) over ALL S*N mask channels (conv_tasnet.py:345-357 quirk): logits first, then one normalising pass
    StageTimer tm(CTN_ST_MASK, st);
    a.mask_logits = 1;
    a.mask_out = nullptr;
    CTN_TRY(pw_dispatch(a, PRO_PRELU, EPI_MASK, mask_math, st));
    return ctn_softmax_mask(ws->what, ws->w, mask_out, B, S * N, N, frames, pitch, st);
  }
  if (dec && !mask_out && mask_math == CTN_MATH_F16X3 && c->kernel_size == 16 && c->stride == 8) {
    PwArgs f = a;
    f.D = dec->out; f.dec_w = p->dec_w; f.dec_crop_left = dec->crop_left; f.dec_T_out = dec->T_out;
    if (ctn_pw_tma_supported(f, PRO_PRELU, EPI_MASKDEC)) {
      StageTimer tm(CTN_ST_MASK, st);
      cudaError_t e = cudaMemsetAsync(dec->out, 0, sizeof(float) * (size_t)B * S * dec->T_out, st);  // tile seams are red.add'ed
      if (e != cudaSuccess) return (int)e;
      CTN_TRY(ctn_pw_tma(f, PRO_PRELU, EPI_MASKDEC, st));
      dec->fused = true;
      return CTN_OK;
    }
  }
  { StageTimer tm(CTN_ST_MASK, st); CTN_TRY(pw_dispatch(a, PRO_PRELU, EPI_MASK, mask_math, st)); }
  return CTN_OK;
}

extern "C" int ctn_convtasnet_fwd(const ctn_config_t* cfg, const ctn_params_t* params, const float* x, int B, int T,
                                  float* out, float* latent, void* workspace, size_t workspace_bytes, ctn_stream_t stream) {
  LaunchScope scope(x);
  CTN_TRY(check_model_cfg(cfg));
  if (!params || !params->blocks || !x || !out || !workspace || B <= 0 || T <= 0) return CTN_EINVAL;
  if (((uintptr_t)workspace) & 255) return CTN_EALIGN;
  size_t need = 0;
  CTN_TRY(ctn_workspace_bytes(cfg, B, T, &need));
  if (workspace_bytes < need) return CTN_EWORKSPACE;
  int pl = 0, pr = 0;
  const int frames = ctn_frames(T, cfg->kernel_size, cfg->stride, &pl, &pr);
  if (frames <= 0) return CTN_EINVAL;
  const int pitch = ctn_pitch(frames);
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(workspace);
  ModelWs ws;
  carve_model(cv, cfg, B, pitch, &ws);
  cudaError_t e = cudaMemsetAsync(ws.stats0, 0, sizeof(double) * 2 * B, st);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(ws.tcn.stats, 0, ws.tcn.stats_bytes, st);
  if (e != cudaSuccess) return (int)e;
  const int Cin = cfg->in_channels > 1 ? cfg->in_channels : 1;  // x (B,Cin,T), out (B,S,Cin,T): conv_tasnet.py:138-141,167-168
  // encoder (+ gLN0 statistics)
  { StageTimer tm(CTN_ST_ENC, st);
    if (Cin == 1) {
      CTN_TRY(ctn_encoder_fwd(x, params->enc_w, ws.w, B, T, pl, pr, cfg->n_basis, cfg->kernel_size, cfg->stride, cfg->enc_relu,
                              pitch, ws.stats0, st));
    } else {
      CTN_TRY(ctn_encoder_mc_fwd(x, params->enc_w, ws.w, B, Cin, T, pl, pr, cfg->n_basis, cfg->kernel_size, cfg->stride, cfg->enc_relu,
                                 pitch, ws.stats0, st));
    } }
  DecFuse dec{out, pl, T, false};
  CTN_TRY(run_separator(cfg, params, &ws, B, frames, pitch, nullptr, st, (latent || Cin > 1) ? nullptr : &dec));
  if (!dec.fused) {
    // decoder + crop (conv_tasnet.py:163-169)
    StageTimer tm(CTN_ST_DEC, st);
    if (Cin == 1) {
      CTN_TRY(ctn_decoder_fwd(ws.what, params->dec_w, out, B * cfg->n_sources, cfg->n_basis, frames, pitch, cfg->kernel_size,
                              cfg->stride, pl, T, st));
    } else {
      CTN_TRY(ctn_decoder_mc_fwd(ws.what, params->dec_w, out, B * cfg->n_sources, Cin, cfg->n_basis, frames, pitch, cfg->kernel_size,
                                 cfg->stride, pl, T, st));
    }
  }
  if (latent) CTN_TRY(ctn_copy_from_pitch(ws.what, latent, B * cfg->n_sources * cfg->n_basis, frames, pitch, st));
  return CTN_OK;
}

// stats of an already-encoded w in padded layout
__global__ void __launch_bounds__(256) k_stats_pitch(const float* __restrict__ x, int C, int frames, int pitch, double* __restrict__ stats) {
  __shared__ double red[64];
  const int b = blockIdx.y;
  double s = 0.0, ss = 0.0;
  for (int c = blockIdx.x; c < C; c += gridDim.x) {
    const float* r = x + ((size_t)b * C + c) * pitch;
    float ls = 0.f, lss = 0.f;
    for (int t = threadIdx.x; t < frames; t += 256) { const float v = r[t]; ls += v; lss += v * v; }
    s += ls; ss += lss;
  }
  block_sum2_d(s, ss, red);
  if (threadIdx.x == 0) { atomicAdd(&stats[2 * b], s); atomicAdd(&stats[2 * b + 1], ss); }
}

extern "C" int ctn_separator_fwd(const ctn_config_t* cfg, const ctn_params_t* params, const float* w, int B, int frames,
                                 float* mask, void* workspace, size_t workspace_bytes, ctn_stream_t stream) {
  LaunchScope scope(w);
  CTN_TRY(check_model_cfg(cfg));
  if (!params || !params->blocks || !w || !mask || !workspace || B <= 0 || frames <= 0) return CTN_EINVAL;
  if (((uintptr_t)workspace) & 255) return CTN_EALIGN;
  const int pitch = ctn_pitch(frames);
  Carver cv0(nullptr);
  ModelWs ws;
  carve_model(cv0, cfg, B, pitch, &ws);
  const size_t mask_elems = (size_t)B * cfg->n_sources * cfg->n_basis * pitch;
  if (workspace_bytes < cv0.off + 512 + mask_elems * sizeof(float)) return CTN_EWORKSPACE;
  Carver cv(workspace);
  carve_model(cv, cfg, B, pitch, &ws);
  float* mask_p = cv.take<float>(mask_elems);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(ws.stats0, 0, sizeof(double) * 2 * B, st);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(ws.tcn.stats, 0, ws.tcn.stats_bytes, st);
  if (e != cudaSuccess) return (int)e;
  CTN_TRY(ctn_copy_to_pitch(w, ws.w, B * cfg->n_basis, frames, pitch, st));
  int gx = cfg->n_basis < 64 ? cfg->n_basis : 64;
  k_stats_pitch<<<dim3(gx, B), 256, 0, st>>>(ws.w, cfg->n_basis, frames, pitch, ws.stats0);
  CTN_COUNT_LAUNCH();
  CTN_RETURN_IF_CUDA_ERR();
  CTN_TRY(run_separator(cfg, params, &ws, B, frames, pitch, mask_p, st));
  CTN_TRY(ctn_copy_from_pitch(mask_p, mask, B * cfg->n_sources * cfg->n_basis, frames, pitch, st));
  return CTN_OK;
}

// ------------------------------------------------------------------------------------------------
// separator stages on the pitched layout (used by the DPRNN-TasNet path, whose dual-path blocks run between them)
// ------------------------------------------------------------------------------------------------
struct StageWs { FoldedConv head; float* wimg; };
static void carve_stage(Carver& cv, int M, int K, int math, StageWs* ws) {
  ws->head.Wf = cv.take<float>((size_t)M * K);
  ws->head.v1 = cv.take<float>(M);
  ws->head.v2 = cv.take<float>(M);
  ws->head.vb = nullptr;
  ws->wimg = math != CTN_MATH_FP32 ? cv.take<float>(ctn_umma_wimg_bytes(M, K, math) / sizeof(float)) : nullptr;
}
extern "C" size_t ctn_stage_workspace_bytes(int M, int K) {
  if (M <= 0 || K <= 0) return 0;
  Carver cv(nullptr);
  StageWs ws;
  carve_stage(cv, M, K, CTN_MATH_TF32X3, &ws);
  return cv.off + 512;
}

// Separator head (src/models/conv_tasnet.py:370-371 == src/models/dprnn_tasnet.py:335-336): x0 = Wb gLN(w) + bb with the gLN
// folded into the contraction.  w (B, N, pitch) pitched, stats0 = double[B][2] (sum, sumsq) of w over its valid frames (as
// ctn_encoder_fwd leaves them); x0 (B, Bc, pitch) pitched.  The operand is un-normalised: fp16-piece mode runs on tf32 pieces.
extern "C" int ctn_sep_head_fwd(const float* w, const double* stats0, const float* norm_g, const float* norm_b, const float* bn_w,
                                const float* bn_b, float* x0, int B, int N, int Bc, int frames, int pitch, float eps, int math,
                                void* workspace, size_t workspace_bytes, ctn_stream_t stream) {
  LaunchScope scope(w);
  if (!w || !stats0 || !norm_g || !norm_b || !bn_w || !x0 || !workspace || B <= 0 || N <= 0 || Bc <= 0 || frames <= 0) return CTN_EINVAL;
  if (pitch < frames || pitch % CTN_TILE_T != 0 || (((uintptr_t)workspace) & 255)) return CTN_EALIGN;
  if (workspace_bytes < ctn_stage_workspace_bytes(Bc, N)) return CTN_EWORKSPACE;
  if (math == CTN_MATH_F16X3) math = CTN_MATH_TF32X3;
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(workspace);
  StageWs ws;
  carve_stage(cv, Bc, N, math, &ws);
  CTN_TRY(ctn_fold_conv(bn_w, bn_b, norm_g, norm_b, Bc, N, ws.head, 0, st));
  PwArgs a;
  memset(&a, 0, sizeof(a));
  a.A = w; a.W = ws.head.Wf; a.D = x0; a.B = B; a.M = Bc; a.K = N; a.frames = frames; a.pitch = pitch;
  a.v1 = ws.head.v1; a.v2 = ws.head.v2; a.stats_in = stats0; a.n_in = (double)N * (double)frames; a.eps = eps;
  if (math != CTN_MATH_FP32) {
    CTN_TRY(ctn_umma_build_wimg(ws.head.Wf, Bc, N, math, ws.wimg, st));
    a.wimg = ws.wimg;
  }
  return pw_dispatch(a, PRO_NONE, EPI_HEAD, math, st);
}

// Separator tail + decoder (conv_tasnet.py:373-376, 158-169 == dprnn_tasnet.py:348-350 + 141-153): PReLU -> mask 1x1 -> sigmoid ->
// w * mask -> ConvTranspose1d -> crop.  y (B, Bc, pitch), w (B, N, pitch) pitched; out (B, S, T) contiguous; latent (nullable)
// (B, S, N, frames) contiguous; what: (B, S*N, pitch) scratch for w_hat.
extern "C" int ctn_sep_tail_fwd(const float* y, const float* w, const float* prelu, const float* mask_w, const float* mask_b,
                                const float* dec_w, float* out, float* latent, float* what, int B, int N, int Bc, int S, int frames,
                                int pitch, int L, int stride, int crop_left, int T, int math, void* workspace, size_t workspace_bytes,
                                ctn_stream_t stream) {
  LaunchScope scope(y);
  if (!y || !w || !prelu || !mask_w || !mask_b || !dec_w || !out || !what || !workspace || B <= 0 || N <= 0 || Bc <= 0 || S <= 0 || frames <= 0)
    return CTN_EINVAL;
  if (pitch < frames || pitch % CTN_TILE_T != 0 || (((uintptr_t)workspace) & 255)) return CTN_EALIGN;
  if (workspace_bytes < ctn_stage_workspace_bytes(S * N, Bc)) return CTN_EWORKSPACE;
  if (math == CTN_MATH_F16X3) math = CTN_MATH_TF32X3;  // un-normalised operand without a static bound: tf32 pieces
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(workspace);
  StageWs ws;
  carve_stage(cv, S * N, Bc, math, &ws);
  PwArgs a;
  memset(&a, 0, sizeof(a));
  a.A = y; a.W = mask_w; a.D = what; a.B = B; a.M = S * N; a.K = Bc; a.frames = frames; a.pitch = pitch;
  a.pro_slope = prelu; a.bias = mask_b; a.wenc = w; a.Nb = N;
  if (math != CTN_MATH_FP32) {
    CTN_TRY(ctn_umma_build_wimg(mask_w, S * N, Bc, math, ws.wimg, st));
    a.wimg = ws.wimg;
  }
  CTN_TRY(pw_dispatch(a, PRO_PRELU, EPI_MASK, math, st));
  CTN_TRY(ctn_decoder_fwd(what, dec_w, out, B * S, N, frames, pitch, L, stride, crop_left, T, stream));
  if (latent) CTN_TRY(ctn_copy_from_pitch(what, latent, B * S * N, frames, pitch, st));
  return CTN_OK;
}

// ------------------------------------------------------------------------------------------------
// end-to-end with host buffers
// ------------------------------------------------------------------------------------------------
struct HostIo {
  float *x, *tgt, *out, *loss_b, *loss_mean;
  int64_t* perm;
  double* scratch;
};
static void carve_io(Carver& cv, const ctn_config_t* c, int B, int T, HostIo* io) {
  const int S = c->n_sources;
  io->x = cv.take<float>((size_t)B * T);
  io->tgt = cv.take<float>((size_t)B * S * T);
  io->out = cv.take<float>((size_t)B * S * T);
  io->loss_b = cv.take<float>(B);
  io->loss_mean = cv.take<float>(1);
  io->perm = cv.take<int64_t>((size_t)B * S);
  io->scratch = cv.take<double>(ctn_sisdr_pit_scratch_bytes(B, S) / sizeof(double));
}

extern "C" size_t ctn_host_io_bytes(const ctn_config_t* cfg, int B, int T) {
  if (!cfg || B <= 0 || T <= 0) return 0;
  Carver cv(nullptr);
  HostIo io;
  carve_io(cv, cfg, B, T, &io);
  return cv.off + 256;
}

extern "C" int ctn_convtasnet_loss_host(const ctn_config_t* cfg, const ctn_params_t* params, const float* x_host,
                                        const float* tgt_host, int B, int T, float* out_host, float* loss_mean_host,
                                        int64_t* perm_host, void* dev_io, size_t dev_io_bytes, void* workspace,
                                        size_t workspace_bytes, float loss_eps, ctn_stream_t stream) {
  LaunchScope scope(dev_io);
  if (cfg && cfg->in_channels > 1) return CTN_EUNSUPPORTED;  // host-buffer entry: monaural mixtures
  if (!cfg || !x_host || !tgt_host || !loss_mean_host || !perm_host || !dev_io || B <= 0 || T <= 0) return CTN_EINVAL;
  if (((uintptr_t)dev_io) & 255) return CTN_EALIGN;
  if (dev_io_bytes < ctn_host_io_bytes(cfg, B, T)) return CTN_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int S = cfg->n_sources;
  Carver cv(dev_io);
  HostIo io;
  carve_io(cv, cfg, B, T, &io);
  cudaError_t e;
  if ((e = cudaMemcpyAsync(io.x, x_host, sizeof(float) * (size_t)B * T, cudaMemcpyHostToDevice, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemcpyAsync(io.tgt, tgt_host, sizeof(float) * (size_t)B * S * T, cudaMemcpyHostToDevice, st)) != cudaSuccess) return (int)e;
  CTN_TRY(ctn_convtasnet_fwd(cfg, params, io.x, B, T, io.out, nullptr, workspace, workspace_bytes, stream));
  CTN_TRY(ctn_sisdr_pit_fwd(io.out, io.tgt, B, S, T, loss_eps, io.loss_b, io.perm, io.loss_mean, nullptr, io.scratch, stream));
  if (out_host && (e = cudaMemcpyAsync(out_host, io.out, sizeof(float) * (size_t)B * S * T, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemcpyAsync(loss_mean_host, io.loss_mean, sizeof(float), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemcpyAsync(perm_host, io.perm, sizeof(int64_t) * (size_t)B * S, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)e;
  return CTN_OK;
}
