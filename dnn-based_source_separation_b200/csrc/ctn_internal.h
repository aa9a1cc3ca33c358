// Internal (non-ABI) declarations shared by the .cu translation units.
#pragma once
#include "ctn_common.cuh"

// ---- folded / derived parameters (built per forward by ctn_prep_*; weights may change every step) ----------
// For a 1x1 conv applied to a gLN output,  W (gamma*(u-mu)*rstd + beta) + b  ==  rstd * (W diag(gamma)) u
//   + (b + W beta) - mu*rstd * (W gamma):   Wf = W diag(gamma),  v1 = b + W beta,  v2 = W gamma.
struct FoldedConv {
  float* Wf;  // (M, K)
  float* v1;  // (M)
  float* v2;  // (M)
  float* vb;  // (M) nullable: bound of |W gLN(u) + b| per row = sum_k |W[m][k]| (|gamma_k| R + |beta_k|) + |b_m|, R = sqrt(#elements
              // of the gLN group) >= max |normalised value|  (activation envelope of the fp16-piece mode)
};

#define CTN_MAX_BLOCKS 64
// epilogue / prologue selectors of the pointwise (1x1) contraction kernels
enum { PRO_NONE = 0, PRO_PRELU = 1, PRO_DW = 2, PRO_RES = 3 };
enum { EPI_RAW = 0, EPI_HEAD = 1, EPI_H = 2, EPI_MASK = 3, EPI_MASKDEC = 4 };

struct PwArgs {
  const float* A;      // (B, K, pitch) activations
  const float* W;      // (M, K) row-major weights
  float* D;            // (B, M, pitch)
  int B, M, K, frames, pitch;
  // prologue
  const float* pro_slope;  // PRO_PRELU / PRO_DW: PReLU slope (1)
  // PRO_DW (tcgen05 path): A is h (B,K,pitch); the producer computes u = PReLU(dwconv3(gLN1(h)) + bd) on the fly
  const float* dw_norm_g;  // (K) gLN1 gamma
  const float* dw_norm_b;  // (K) gLN1 beta
  const float* dw_w;       // (K,3) depthwise taps
  const float* dw_b;       // (K)
  const double* dw_stats_in;   // (B,2) (sum, sumsq) of h
  double* dw_stats_out;        // (B,2) += (sum, sumsq) of u
  int dw_dilation, dw_pad_left;
  float dw_eps;
  // epilogue
  const float* bias;       // EPI_H / EPI_MASK: (M)
  const float* slope;      // EPI_H: PReLU slope (1)
  const float* v1;         // EPI_HEAD
  const float* v2;         // EPI_HEAD
  const double* stats_in;  // EPI_HEAD: (B,2) of the input tensor
  double n_in;             // EPI_HEAD: element count of a gLN group of the input
  float eps;               // EPI_HEAD
  double* stats_out;       // EPI_H: (B,2) += (sum, sumsq) over valid outputs
  int store_pre;           // EPI_H (tcgen05 path only): store W A + bias (pre-activation) instead of PReLU(.); stats unchanged
  const float* wenc;       // EPI_MASK: encoder output (B, Nb, pitch)
  int Nb;                  // EPI_MASK: n_basis
  float* mask_out;         // EPI_MASK: optional raw mask output (B, M, pitch)
  int mask_logits;         // EPI_MASK: 1 = store the LOGITS (W A + bias) to D, no sigmoid, no w product (softmax masks take a second pass)
  // EPI_MASKDEC (TMA-fed kernel): mask 1x1 + sigmoid + w*mask + transposed-conv decoder + crop in one epilogue; w_hat is never
  // materialised.  D = estimates (B, M/Nb, dec_T_out) contiguous, ZERO-initialised by the caller (tile seams are red.add'ed)
  const float* dec_w;      // (Nb, 1, 16) decoder basis, kernel 16 / stride 8
  int dec_crop_left, dec_T_out;
  // PRO_RES (tcgen05 path): the operand is the UPDATED residual stream  x_new = A + rstd*res_r[:K] + (v1 - mean*rstd*v2)
  // (the deferred gLN2 of the previous block); CTAs with n-tile 0 also store x_new to res_x_out (ping-pong buffer).
  const float* res_r;       // (B, res_Mt, pitch) raw [out;skip] contraction of the previous block; rows [0,K) are used
  int res_Mt;
  const float* res_v1;      // (>=K) folded bias vectors of the previous block
  const float* res_v2;
  const double* res_stats;  // (B,2) stats2 of the previous block
  double res_n;
  float res_eps;
  float* res_x_out;         // (B, K, pitch)
  // tcgen05 path only
  const float* wimg;       // pre-swizzled hi/lo weight images (ctn_umma_build_wimg)
  // fp16-piece mode: power-of-two scale of the activation operand (device scalar, nullable = 1), chosen per forward from a
  // bound on |operand| derived from the weights alone (ctn_act_scales) so that fp16 can never saturate; undone in the epilogue
  const float* act_scale;
  const float* dw_params;  // PRO_DW, TMA-fed kernel: packed per-channel parameters [ceil16(K)][8] (ctn_act_scales)
  // PRO_DW, training forward (TMA-fed kernel): A holds the PRE-activation h_pre = W1 x + b1 (the backward needs it), the producer
  // applies PReLU(dw_in_slope) on load; the depthwise pre-activation u_pre is stored to dw_u_pre_out (B, K, pitch)
  const float* dw_in_slope;
  float* dw_u_pre_out;
};

// Output channels per n-tile (UMMA N) of the tcgen05 pointwise kernels.  The weight images are laid out in n-tiles of this width,
// so the image builders and both kernel families use this one rule.
__host__ __device__ inline int pick_n_tile(int M) { return M >= 256 ? 256 : ((M + 15) / 16) * 16; }
// the fp16-piece mode keeps one scale per padded output channel in shared memory: contractions with more than
// CTN_F16_MAX_ROWS padded output channels use the tf32 pieces instead (images and kernel are chosen by the same rule)
constexpr int CTN_F16_MAX_ROWS = 2048;
__host__ __device__ inline int eff_math(int M, int math) {
  if (math != CTN_MATH_F16X3) return math;
  const int n_tile = pick_n_tile(M);
  return ((M + n_tile - 1) / n_tile) * n_tile > CTN_F16_MAX_ROWS ? CTN_MATH_TF32X3 : math;
}

// fp32 CUDA-core path (ctn_tcn_simt.cu)
int ctn_pw_simt(const PwArgs& a, int pro, int epi, cudaStream_t st);
// tcgen05 path (ctn_umma.cu); math = CTN_MATH_TF32X3 / CTN_MATH_TF32
int ctn_pw_umma(const PwArgs& a, int pro, int epi, int math, cudaStream_t st);
size_t ctn_umma_wimg_bytes(int M, int K, int math);
int ctn_umma_build_wimg(const float* W, int M, int K, int math, float* wimg, cudaStream_t st);

// tcgen05 weight gradient of a 1x1 conv (ctn_wgrad_umma.cu): dW (M,K) += sum_{b,t} dY[b][m][t] X[b][k][t]; rows
// [0,split_row) -> dWa, rest -> dWb (nullable).  dW must be zero-initialised by the caller (split-K partials are added).
int ctn_wgrad_umma(const float* dy, size_t dy_bs, const float* x, size_t x_bs, float* dWa, float* dWb, int split_row, int M,
                   int K, int B, int frames, int pitch, int math, cudaStream_t st);

int ctn_fold_conv(const float* W, const float* bias, const float* gamma, const float* beta, int M, int K, FoldedConv out,
                  int row_offset, cudaStream_t st, float R = 0.f);

// batched variants: all weight preparation of a forward in two launches (jobs travel in the kernel parameter block)
struct FoldJob { const float *W, *bias, *gamma, *beta; float *Wf, *v1, *v2; int M, K, row_offset; float* vb; float R; };
struct WimgJob { const float* W; float* wimg; int M, K; };
#define CTN_MAX_JOBS 48
int ctn_fold_batch(const FoldJob* jobs, int n, cudaStream_t st);
int ctn_umma_build_wimg_batch(const WimgJob* jobs, int n, int math, cudaStream_t st);

// TMA-fed tcgen05 kernels of the fp16-piece mode (ctn_pwtma.cu): pw1 (PRO_RES / PRO_NONE + EPI_H) and pw2 (PRO_DW + EPI_RAW)
int ctn_pw_tma_supported(const PwArgs& a, int pro, int epi);
int ctn_pw_tma(const PwArgs& a, int pro, int epi, cudaStream_t st);

// Activation envelope of the fp16-piece mode.  Per residual block i the two operands that meet the tensor core as fp16
// pieces are x_i (pw1) and u_i (fused depthwise output, pw2); the mask contraction sees PReLU(skip sum).  From the weights
// alone:  |gLN(.)| <= |gamma| R + |beta| with R = sqrt(#elements of the group);  |u_c| <= max(1,|a2|) ((|g1_c| R + |b1_c|) sum_k |wd_ck| + |bd_c|);
// |x_{i+1}| <= |x_i| + max_n vb_out_i[n];  |skip| <= sum_i max_n vb_skip_i[n].  scales[2i] / [2i+1] / [2n] receive the powers of two
// that map those bounds to <= 2^15; dwp_i receives the packed depthwise parameters {g1, b1, w0, w1, w2, bd, 0, 0} per channel.
struct ScaleJob { const float *vb, *g1, *b1, *dw_w, *dw_b, *slope2; float* dwp; int has_out; };
struct ScaleJobs {
  ScaleJob j[CTN_MAX_BLOCKS];
  int n, Bc, Sc, H, P;
  const float* x0_bound;  // device: x0_n candidates whose max bounds |x_0|
  int x0_n;
  const float* mask_slope;  // nullable
  float R;
  float* scales;  // [2n + 1]
};
int ctn_act_scales(const ScaleJobs& jobs, cudaStream_t st);
// max |x| over rows x frames of a pitched tensor -> *out (float, must be zeroed by the caller)
int ctn_absmax_pitch(const float* x, int rows, int frames, int pitch, float* out, cudaStream_t st);

// training forward of the TCN through the fused inference kernels (ctn_api.cu); per-block buffers owned by the training workspace
struct TcnTrainHooks { float* const* x_keep; float* const* hpre; float* const* upre; };
size_t ctn_tcn_train_ws_bytes(const ctn_config_t* c, int B, int pitch);
int ctn_tcn_train_fwd(const ctn_config_t* c, const ctn_block_params_t* blocks, void* mem, size_t mem_bytes, const TcnTrainHooks* hooks,
                      double* stats, float* skip, const float* x0_bound, int x0_n, const float* mask_slope, const float** mask_scale,
                      int B, int frames, int pitch, cudaStream_t st);

// mask_nonlinear = 'softmax' (src/models/conv_tasnet.py:345-357, 375-376: nn.Softmax(dim=1) over ALL S*N channels before the view):
// in place on the logits (B, M, pitch): what = softmax_m(logits) * w[m % Nb]; mask_out (nullable) receives the softmax itself
int ctn_softmax_mask(float* logits_what, const float* wenc, float* mask_out, int B, int M, int Nb, int frames, int pitch, cudaStream_t st);

// depthwise stage: u = PReLU(dwconv(gLN1(h))) (+ stats2), all (B,H,pitch)
int ctn_dw_fwd(const float* h, float* u, const float* norm_g, const float* norm_b, const float* dw_w, const float* dw_b,
               const float* slope, const double* stats_in, double* stats_out, int B, int H, int frames, int pitch, int P,
               int dilation, int causal, float eps, cudaStream_t st);

// finishing: x += rstd2*outraw[:Bc] + c ; skip (+)= rstd2*outraw[Bc:] + c
int ctn_finish_fwd(const float* outraw, const FoldedConv f, const double* stats2, double n2, float eps, float* x,
                   float* skip, int B, int Bc, int Sc, int has_out, int skip_init, int frames, int pitch, cudaStream_t st);

// deferred skip reduction: skip[b][m][t] = sum_i ( rstd2_i[b] * r_i[b][off_i + m][t] + (v1_i[off_i+m] - mean_i rstd_i v2_i[off_i+m]) )
// over all residual blocks i -- reads every block's skip rows ONCE instead of read-modify-writing the accumulator per block
struct SkipJob { const float* r; const float* v1; const float* v2; const double* stats2; int off; int Mt; };
struct SkipJobs { SkipJob j[CTN_MAX_BLOCKS]; int n; };
int ctn_skip_reduce(const SkipJobs& jobs, double n2, float eps, float* skip, int B, int Sc, int frames, int pitch, cudaStream_t st);

int ctn_copy_to_pitch(const float* src, float* dst, int rows, int frames, int pitch, cudaStream_t st);
int ctn_copy_from_pitch(const float* src, float* dst, int rows, int frames, int pitch, cudaStream_t st);

// cLN (src/modules/norm.py:78-90) on the padded (B, C, pitch) layout, in place allowed; scratch double[B][frames][2]
int ctn_cln_pitch_fwd(const float* x, const float* gamma, const float* beta, float* y, int B, int C, int frames, int pitch,
                      float eps, double* scratch, cudaStream_t st);

// Causal (cLN) models: un-fused pipeline in the reference's operation order (ctn_causal.cu).  The cumulative statistics of
// cLN depend on every earlier frame, so the gLN tricks of the fused stack (statistics from the producing epilogue, affine
// folded into the next contraction) do not apply; each block is contraction -> cLN -> causal depthwise -> cLN -> contraction.
size_t ctn_causal_ws_bytes(const ctn_config_t* c, int B, int pitch);
// x: (B, Bc, pitch) block-0 input (updated in place); skip: (B, Sc, pitch) result; h, u: (B, H, pitch) scratch
int ctn_causal_tcn(const ctn_config_t* c, const ctn_block_params_t* blocks, float* x, float* skip, float* h, float* u, int B,
                   int frames, int pitch, void* cws, cudaStream_t st);
// separator head for causal models: x0 = Wb cLN0(w) + bb;  tmp: (B, N, pitch) scratch
int ctn_causal_head(const ctn_config_t* c, const ctn_params_t* p, const float* w, float* tmp, float* x0, int B, int frames,
                    int pitch, void* cws, cudaStream_t st);
