/* ctn_b200.h -- C ABI of the B200-native Conv-TasNet separation path.
 *
 * The reference (tky823/DNN-based_source_separation) has NO native/FFI layer: the path sits behind
 * Python nn.Module classes (SURVEY.md section 8b).  This header is therefore the boundary a maintainer would
 * bind from those classes (ctypes stub shown in INTEGRATION.md).  Each entry point names the reference
 * interface it replaces (file:line relative to the reference root).
 *
 * Conventions
 *   - plain C types only; device pointers are raw `float*` / `int64_t*`; `ctn_stream_t` is a cudaStream_t.
 *   - every call is asynchronous on `stream`, never allocates or frees, never retains pointers.
 *   - return 0 on success, negative CTN_E* for argument / envelope errors, positive = cudaError_t.
 *   - activations inside the library use (batch, channels, pitch) fp32 with pitch = ctn_pitch(frames)
 *     (frames rounded up to 128) so every row is 512-byte aligned; tensors crossing the boundary are
 *     PyTorch-contiguous.
 *   - there is no CPU fallback.  Unsupported configurations return CTN_EUNSUPPORTED.
 */
#ifndef CTN_B200_H
#define CTN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* ctn_stream_t; /* cudaStream_t */

#define CTN_VERSION 100 /* 0.1.0 */

enum ctn_status {
  CTN_OK = 0,
  CTN_EINVAL = -1,       /* bad shape / null pointer              -> Python ValueError        */
  CTN_EUNSUPPORTED = -2, /* outside the kernel envelope           -> Python NotImplementedError */
  CTN_EALIGN = -3,       /* pointer / pitch alignment             -> Python ValueError        */
  CTN_EWORKSPACE = -4,   /* workspace too small                   -> Python RuntimeError      */
  CTN_ENOTBUILT = -5     /* kernel family not compiled into lib   -> Python RuntimeError      */
};

/* numeric mode of the dense 1x1 contractions */
enum ctn_math {
  CTN_MATH_FP32 = 0,   /* CUDA-core FFMA, exact fp32 products (verification mode)          */
  CTN_MATH_TF32X3 = 1, /* tcgen05 kind::tf32, 3-pass hi/lo split, fp32 accumulate (default) */
  CTN_MATH_TF32 = 2,   /* tcgen05 kind::tf32 single pass (fast mode, looser tolerance)      */
  CTN_MATH_F16X3 = 3   /* tcgen05 kind::f16, 3-pass fp16 hi/lo split (11-bit pieces like TF32, twice the MMA rate), fp32
                          accumulate; default of the Python classes.  Weight rows are rescaled by powers of two inside the
                          library (any magnitude is fine); activations must stay below 65504 in magnitude (conversion
                          saturates beyond) -- always true behind the normalisations of this network; the separator head
                          (un-normalised encoder output) and all gradient contractions use the TF32 pieces regardless */
};

/* Constructor arguments of ConvTasNet / Separator (src/models/conv_tasnet.py:57-66, 322-328). */
typedef struct ctn_config {
  int32_t n_basis;      /* N  */
  int32_t kernel_size;  /* L  */
  int32_t stride;       /* L/2 by default */
  int32_t bottleneck;   /* B  (sep_bottleneck_channels) */
  int32_t hidden;       /* H  (sep_hidden_channels)     */
  int32_t skip;         /* Sc (sep_skip_channels)       */
  int32_t sep_kernel;   /* P  (sep_kernel_size)         */
  int32_t num_blocks;   /* R  */
  int32_t num_layers;   /* X  */
  int32_t n_sources;    /* S  */
  int32_t causal;       /* 0: gLN (supported), 1: cLN (CTN_EUNSUPPORTED in the fused path) */
  int32_t enc_relu;     /* enc_nonlinear == 'relu' */
  int32_t mask_softmax; /* mask_nonlinear == 'softmax' -> CTN_EUNSUPPORTED */
  int32_t math;         /* enum ctn_math */
  float eps;            /* Separator head norm eps (ConvTasNet eps)            */
  float eps_tcn;        /* eps of the norms inside the TDCN (reference passes the default 1e-12) */
  int32_t in_channels;  /* C = n_mics of the 4-D input form (conv_tasnet.py:75,138-141); 0 or 1: monaural.  > 1: forward only */
} ctn_config_t;

/* Parameters of one ResidualBlock1d (+ its DepthwiseSeparableConv1d), src/models/tdcn.py:77-196.
 * state_dict names (prefix separator.tdcn.net.{r}.net.{x}.) are given per field. */
typedef struct ctn_block_params {
  const float* bottleneck_w; /* bottleneck_conv1d.weight (H,B,1)                       */
  const float* bottleneck_b; /* bottleneck_conv1d.bias   (H)                           */
  const float* prelu1;       /* nonlinear1d.weight (1)                                 */
  const float* norm1_g;      /* norm1d.norm.weight (H)                                 */
  const float* norm1_b;      /* norm1d.norm.bias   (H)                                 */
  const float* dw_w;         /* separable_conv1d.depthwise_conv1d.weight (H,1,P)       */
  const float* dw_b;         /* separable_conv1d.depthwise_conv1d.bias   (H)           */
  const float* prelu2;       /* separable_conv1d.nonlinear1d.weight (1)                */
  const float* norm2_g;      /* separable_conv1d.norm1d.norm.weight (H)                */
  const float* norm2_b;      /* separable_conv1d.norm1d.norm.bias   (H)                */
  const float* out_w;        /* separable_conv1d.output_pointwise_conv1d.weight (B,H,1) or NULL (last block) */
  const float* out_b;        /* ...bias (B) or NULL                                    */
  const float* skip_w;       /* separable_conv1d.skip_pointwise_conv1d.weight (Sc,H,1) */
  const float* skip_b;       /* ...bias (Sc)                                           */
} ctn_block_params_t;

typedef struct ctn_params {
  const float* enc_w;      /* encoder.conv1d.weight (N,1,L)                  */
  const float* norm0_g;    /* separator.norm1d.norm.weight (N)               */
  const float* norm0_b;    /* separator.norm1d.norm.bias   (N)               */
  const float* bn_w;       /* separator.bottleneck_conv1d.weight (B,N,1)     */
  const float* bn_b;       /* separator.bottleneck_conv1d.bias   (B)         */
  const ctn_block_params_t* blocks; /* HOST array of R*X entries (device pointers inside) */
  const float* prelu_out;  /* separator.prelu.weight (1)                      */
  const float* mask_w;     /* separator.mask_conv1d.weight (S*N,Sc,1)        */
  const float* mask_b;     /* separator.mask_conv1d.bias   (S*N)             */
  const float* dec_w;      /* decoder.conv_transpose1d.weight (N,1,L)        */
} ctn_params_t;

/* ---- introspection ------------------------------------------------------------------------- */
int ctn_version(void);
const char* ctn_strerror(int status);
/* 1 if the tcgen05 (sm_100a) kernel family is compiled in */
int ctn_has_tcgen05(void);

/* ---- geometry helpers (host only) ----------------------------------------------------------
 * ConvTasNet.extract_latent padding rule, src/models/conv_tasnet.py:145-149. */
int ctn_frames(int T, int kernel_size, int stride, int* pad_left, int* pad_right); /* returns T' or <0 */
int ctn_pitch(int frames);                                                         /* frames rounded up to 128 */
/* bytes of device workspace ctn_convtasnet_fwd needs for (batch, T) */
int ctn_workspace_bytes(const ctn_config_t* cfg, int batch, int T, size_t* bytes);

/* ---- module-level entry points -------------------------------------------------------------- */

/* Encoder.forward, src/models/filterbank.py:222-229 (Conv1d(1,N,L,stride,bias=False) [+ReLU]).
 * x (B,1,T) contiguous; virtual zero padding pad_left/pad_right; w (B,N,w_pitch) with frames valid columns,
 * columns [frames,w_pitch) are written as zero.  stats (nullable): double[B][2] += (sum, sumsq) over valid. */
int ctn_encoder_fwd(const float* x, const float* enc_w, float* w, int B, int T, int pad_left, int pad_right,
                    int N, int L, int stride, int relu, int w_pitch, double* stats, ctn_stream_t stream);

/* Decoder.forward, src/models/filterbank.py:245-247 (ConvTranspose1d(N,1,L,stride,bias=False)), fused with the
 * crop of conv_tasnet.py:169: y[bs][t] = full[bs][t + crop_left], t in [0,T_out).  w_hat (BS,N,in_pitch). */
int ctn_decoder_fwd(const float* w_hat, const float* dec_w, float* y, int BS, int N, int frames, int in_pitch,
                    int L, int stride, int crop_left, int T_out, ctn_stream_t stream);
/* Multichannel filter banks, src/models/filterbank.py:212,241 with in_channels = C > 1 (the 4-D input of conv_tasnet.py:138-141):
 * x (B,C,T), enc_w (N,C,L) -> w (B,N,w_pitch) [+ gLN statistics]; w_hat (BS,N,in_pitch), dec_w (N,C,L) -> y (BS,C,T_out), cropped. */
int ctn_encoder_mc_fwd(const float* x, const float* enc_w, float* w, int B, int C, int T, int pad_left, int pad_right, int N, int L,
                       int stride, int relu, int w_pitch, double* stats, ctn_stream_t stream);
int ctn_decoder_mc_fwd(const float* w_hat, const float* dec_w, float* y, int BS, int C, int N, int frames, int in_pitch, int L,
                       int stride, int crop_left, int T_out, ctn_stream_t stream);

/* GlobalLayerNorm.forward, src/modules/norm.py:18,32 (GroupNorm(1,C,eps)).  x,y (B,C,T) contiguous.
 * scratch: double[B][2], zero-initialised by the callee. */
int ctn_gln_fwd(const float* x, const float* gamma, const float* beta, float* y, int B, int C, int T, float eps,
                double* scratch, ctn_stream_t stream);

/* CumulativeLayerNorm1d.forward, src/modules/norm.py:78-90.  x,y (B,C,T) contiguous; scratch double[B][T][2]. */
int ctn_cln_fwd(const float* x, const float* gamma, const float* beta, float* y, int B, int C, int T, float eps,
                double* scratch, ctn_stream_t stream);

/* TimeDilatedConvNet.forward == TemporalConvNet.forward, src/models/tdcn.py:29-41 (src/models/tcn.py:37-49).
 * x (B,bottleneck,frames) contiguous -> skip sum (B,skip,frames) contiguous.  Uses cfg fields bottleneck, hidden,
 * skip, sep_kernel, num_blocks, num_layers, causal, math, eps_tcn.  workspace sized by ctn_tcn_workspace_bytes. */
int ctn_tcn_workspace_bytes(const ctn_config_t* cfg, int batch, int frames, size_t* bytes);
int ctn_tcn_fwd(const ctn_config_t* cfg, const ctn_block_params_t* blocks, const float* x, float* skip_out, int B,
                int frames, void* workspace, size_t workspace_bytes, ctn_stream_t stream);

/* ResidualBlock1d.forward (src/models/tdcn.py:107-147, n_blocks = 1) / TimeDilatedConvBlock1d.forward (tdcn.py:65-75): a run of
 * residual blocks with EXPLICIT dilations returning both heads.  x (B,bottleneck,frames) -> x_out (nullable; the residual stream
 * after the last block, which must then have the output head) and skip_out (B,skip,frames) = sum of the blocks' skip heads.
 * cfg as for ctn_tcn_fwd (num_blocks / num_layers are ignored); workspace: ctn_tcn_workspace_bytes with num_blocks = 1,
 * num_layers = n_blocks.  Non-causal (gLN) only. */
int ctn_tcn_blocks_fwd(const ctn_config_t* cfg, const ctn_block_params_t* blocks, int n_blocks, const int* dilations, const float* x,
                       float* x_out, float* skip_out, int B, int frames, void* workspace, size_t workspace_bytes, ctn_stream_t stream);

/* ConvTasNet.forward / extract_latent, src/models/conv_tasnet.py:116-171.
 * x (B,1,T) -> out (B,S,T); latent (nullable) (B,S,N,frames) contiguous. */
int ctn_convtasnet_fwd(const ctn_config_t* cfg, const ctn_params_t* params, const float* x, int B, int T, float* out,
                       float* latent, void* workspace, size_t workspace_bytes, ctn_stream_t stream);

/* Separator.forward, src/models/conv_tasnet.py:359-378: w (B,N,frames) -> mask (B,S,N,frames), both contiguous. */
int ctn_separator_fwd(const ctn_config_t* cfg, const ctn_params_t* params, const float* w, int B, int frames,
                      float* mask, void* workspace, size_t workspace_bytes, ctn_stream_t stream);

/* ---- DPRNN-TasNet path (BASELINE cfg4): segment / dual-path glue / overlap-add, and the separator stages around it ----
 *
 * Segment1d.forward, src/models/transform.py:15-29, fused with the zero padding of src/models/dprnn_tasnet.py:339-345:
 * x (B,F,pitch) with `frames` valid columns (pitch == frames for a contiguous tensor) -> chunks of `chunk_size` frames every
 * `hop_size` of the padded sequence, S = (frames + pad_left + pad_right - chunk_size) / hop_size + 1.
 * channels_last = 0: Z (B,F,S,chunk) -- the reference layout;  1: Z (B,S,chunk,F) -- the batch_first layout the intra-chunk
 * LSTM consumes, i.e. the permute of src/models/dprnn.py:83-84 folded in. */
int ctn_segment_fwd(const float* x, float* Z, int B, int F, int frames, int pitch, int chunk_size, int hop_size, int pad_left,
                    int pad_right, int channels_last, ctn_stream_t stream);
/* OverlapAdd1d.forward, src/models/transform.py:46-62, fused with the crop of dprnn_tasnet.py:347: y (B,F,out_pitch),
 * y[..][t] = sum of the chunks covering padded frame t + crop_left, t < T_out; columns [T_out,out_pitch) = 0.
 * Z laid out as above (channels_last). */
int ctn_overlap_add_fwd(const float* Z, float* y, int B, int F, int S, int chunk_size, int hop_size, int crop_left, int T_out,
                        int out_pitch, int channels_last, ctn_stream_t stream);
/* Tail of IntraChunkRNN / InterChunkRNN.forward, src/models/dprnn.py:87-94 / 140-148: out = gLN(Y; gamma, beta) + R on
 * channels-last tensors (B,D1,D2,F) (gLN = GroupNorm(1,F): per-sample statistics over D1*D2*F values).  swap = 1 stores out as
 * (B,D2,D1,F) -- the layout of the other path (the permutes of dprnn.py:83, 91, 136, 144-146).  scratch: double[B][2]. */
int ctn_dprnn_norm_res_fwd(const float* Y, const float* R, const float* gamma, const float* beta, float* out, int B, int D1, int D2,
                           int F, float eps, int swap, double* scratch, ctn_stream_t stream);
/* Bidirectional LSTM + the 2H -> F Linear of a dual-path block, src/models/dprnn.py:85-87 / 138-139 (nn.LSTM(batch_first,
 * bidirectional) followed by nn.Linear), on tcgen05 with h resident in tensor memory (csrc/ctn_lstm.cu).
 * z (NSEQ,T,F) fp32, batch_first; w[8] = host array of device pointers in torch.nn.LSTM order: weight_ih_l0 (4H,F), weight_hh_l0
 * (4H,H), bias_ih_l0, bias_hh_l0 (4H), then the four *_reverse tensors; gate order i,f,g,o; zero initial state.
 * w_fc (Fo,2H) nullable.  P (2,NSEQ,T,Fo): partial projections W_fc[:, dir*H:(dir+1)*H] h_dir WITHOUT the Linear's bias -- the
 * Linear output is P[0] + P[1] + bias (ctn_dprnn_norm_res2_fwd consumes it in that form).  hout (NSEQ,T,2H) nullable: the LSTM
 * output itself (forward direction in [:H], reverse in [H:]).  Envelope: F, H in {32,64,128}, Fo in {32,64,96,128}
 * (ctn_bilstm_supported); workspace >= ctn_bilstm_workspace_bytes(F,H,Fo), 256-byte aligned.  z_absmax (nullable): device word holding
 * the bit pattern of max|z| (the fp16 operand scale of x is derived from it); null = measured here with one more pass over z. */
int ctn_bilstm_supported(int F, int H, int Fo);
int ctn_debug_lstm_timeline(unsigned long long* out, int n); /* debug: cycle stamps of one CTA (CTN_LSTM_DBG=16), tools/lstm_time.py */
size_t ctn_bilstm_workspace_bytes(int F, int H, int Fo);
int ctn_bilstm_proj_fwd(const float* z, int NSEQ, int T, int F, int H, const float* const* w, const float* w_fc, int Fo, float* P,
                        float* hout, const unsigned* z_absmax, void* workspace, size_t workspace_bytes, ctn_stream_t stream);
/* ctn_dprnn_norm_res_fwd with Y = P[0] + P[1] + fc_bias, P (2,B,D1,D2,F) as ctn_bilstm_proj_fwd leaves it (F % 4 == 0).
 * out_absmax (nullable): receives the bit pattern of max|out| -- the z_absmax of the next ctn_bilstm_proj_fwd. */
int ctn_dprnn_norm_res2_fwd(const float* P, const float* fc_bias, const float* R, const float* gamma, const float* beta, float* out,
                            int B, int D1, int D2, int F, float eps, int swap, double* scratch, unsigned* out_absmax, ctn_stream_t stream);
/* Separator head on the padded layout, src/models/conv_tasnet.py:370-371 == src/models/dprnn_tasnet.py:335-336:
 * x0 (B,Bc,pitch) = Wb gLN(w) + bb; w (B,N,pitch), stats0 double[B][2] = (sum, sumsq) of w (as ctn_encoder_fwd leaves them).
 * workspace >= ctn_stage_workspace_bytes(Bc, N). */
size_t ctn_stage_workspace_bytes(int M, int K);
int ctn_sep_head_fwd(const float* w, const double* stats0, const float* norm_g, const float* norm_b, const float* bn_w,
                     const float* bn_b, float* x0, int B, int N, int Bc, int frames, int pitch, float eps, int math, void* workspace,
                     size_t workspace_bytes, ctn_stream_t stream);
/* Separator tail + decoder, conv_tasnet.py:373-376,158-169 == dprnn_tasnet.py:348-350,141-153: PReLU -> mask 1x1 -> sigmoid ->
 * w*mask -> ConvTranspose1d -> crop.  y (B,Bc,pitch), w (B,N,pitch); out (B,S,T); latent nullable (B,S,N,frames);
 * what (B,S*N,pitch) scratch; workspace >= ctn_stage_workspace_bytes(S*N, Bc). */
int ctn_sep_tail_fwd(const float* y, const float* w, const float* prelu, const float* mask_w, const float* mask_b,
                     const float* dec_w, float* out, float* latent, float* what, int B, int N, int Bc, int S, int frames, int pitch,
                     int L, int stride, int crop_left, int T, int math, void* workspace, size_t workspace_bytes, ctn_stream_t stream);

/* modules.conv.DepthwiseSeparableConv1d.forward, src/modules/conv.py:24-28 (not on Conv-TasNet's path; API completeness).
 * Depthwise stage: x (B,C,T) contiguous, w (C,1,K), bias nullable -> y (B,C,y_pitch) with T_out = (T + 2 padding - dilation (K-1) - 1)
 * / stride + 1 valid columns, the rest zero.  Pointwise stage: x (B,K,pitch) padded layout with `frames` valid columns, W (M,K,1),
 * bias nullable -> y (B,M,frames) contiguous; workspace >= 4*B*M*pitch + ctn_stage_workspace_bytes(M,K) + 16*B + 4096 bytes. */
int ctn_depthwise_conv1d_fwd(const float* x, const float* w, const float* bias, float* y, int B, int C, int T, int K, int stride, int padding,
                             int dilation, int y_pitch, ctn_stream_t stream);
int ctn_pointwise_conv1d_fwd(const float* x, const float* W, const float* bias, float* y, int B, int M, int K, int frames, int pitch,
                             int math, void* workspace, size_t workspace_bytes, ctn_stream_t stream);

/* sisdr, src/criterion/sdr.py:122-139: est,tgt (rows,T) contiguous -> out (rows). scratch double[rows][4]. */
int ctn_sisdr_fwd(const float* est, const float* tgt, int rows, int T, float eps, float* out, double* scratch,
                  ctn_stream_t stream);
/* sdr(), src/criterion/sdr.py:6-20: out[r] = 10 log10((|tgt_r|^2 + eps) / (|tgt_r - est_r|^2 + eps)); est, tgt (rows,T) contiguous;
 * scratch: double[rows][2]. */
int ctn_sdr_fwd(const float* est, const float* tgt, int rows, int T, float eps, float* out, double* scratch, ctn_stream_t stream);

/* PIT1d(NegSISDR(reduction='mean')), src/criterion/pit.py:9-44,71-77 + src/criterion/sdr.py:198-227.
 * est,tgt (B,S,T) contiguous.  loss_b (B) = min over permutations of -mean_i SI-SDR(est_i, tgt_perm[i]);
 * perm (B,S) int64, estimate i <-> target perm[i] (first minimum on ties, lexicographic permutation order);
 * loss_mean (1) = mean over the batch.  pair_sisdr (nullable) (B,S,S) = SI-SDR(est_i, tgt_j).
 * scratch: double[B][S*S*2 + S], zero-initialised by the callee.  S <= 6. */
int ctn_sisdr_pit_fwd(const float* est, const float* tgt, int B, int S, int T, float eps, float* loss_b,
                      int64_t* perm, float* loss_mean, float* pair_sisdr, double* scratch, ctn_stream_t stream);
size_t ctn_sisdr_pit_scratch_bytes(int B, int S);

/* End-to-end call with HOST buffers (the "e2e" leg): copies x_host (B,1,T) and tgt_host (B,S,T) (pinned or
 * pageable) to the device staging areas, runs ctn_convtasnet_fwd + ctn_sisdr_pit_fwd, copies back out_host
 * (nullable, (B,S,T)), loss_mean_host (1), perm_host (B,S).  All on `stream`; the caller synchronises.
 * dev_io: device staging of dev_io_bytes >= ctn_host_io_bytes() (checked); loss_eps: eps of the SI-SDR (sdr.py:122, 1e-12). */
size_t ctn_host_io_bytes(const ctn_config_t* cfg, int B, int T);
int ctn_convtasnet_loss_host(const ctn_config_t* cfg, const ctn_params_t* params, const float* x_host,
                             const float* tgt_host, int B, int T, float* out_host, float* loss_mean_host,
                             int64_t* perm_host, void* dev_io, size_t dev_io_bytes, void* workspace,
                             size_t workspace_bytes, float loss_eps, ctn_stream_t stream);

/* ---- training path: what `loss.backward()` does in the reference trainer (egs/wsj0-mix/common/src/driver.py:146-150) ----
 * ctn_convtasnet_fwd_train == ctn_convtasnet_fwd (same estimate) but keeps, inside `train_ws`, what the backward needs:
 * encoder output, mask, every residual block's input and the two pre-activations (W1 x + b1, dwconv(..) + bd) and the gLN
 * statistics.  ctn_convtasnet_bwd then turns d_out (B,S,T), the gradient of the estimate, into the gradients of all
 * parameters.  `grads` has the layout of ctn_params_t (same shapes as the parameters); every gradient tensor must be
 * ZERO on entry (kernels accumulate with atomics) and is complete on return.  The gradient w.r.t. the mixture is not
 * produced (the reference trainer never asks for it).  train_ws: ctn_train_workspace_bytes(), 256-byte aligned, must
 * be left untouched between the two calls.  Envelope: non-causal gLN, sigmoid mask, sep_kernel <= 8. */
typedef ctn_params_t ctn_grads_t;
int ctn_train_workspace_bytes(const ctn_config_t* cfg, int batch, int T, size_t* bytes);
int ctn_convtasnet_fwd_train(const ctn_config_t* cfg, const ctn_params_t* params, const float* x, int B, int T, float* out,
                             void* train_ws, size_t train_ws_bytes, ctn_stream_t stream);
int ctn_convtasnet_bwd(const ctn_config_t* cfg, const ctn_params_t* params, const ctn_grads_t* grads, const float* x,
                       const float* d_out, int B, int T, void* train_ws, size_t train_ws_bytes, ctn_stream_t stream);

/* Backward of ctn_sisdr_pit_fwd through the selected permutation (src/criterion/pit.py:36-44; sdr.py:135-137):
 * d_est (B,S,T) = grad_loss_b[b] * coef * dSI-SDR(est_i, tgt_perm[i])/d est_i.  fwd_scratch = the scratch buffer the
 * forward call filled (pair statistics), perm = its permutation output.  grad_loss_b (B) nullable (= 1);
 * coef = -1/S for NegSISDR(reduction='mean'), -1 for 'sum'. */
int ctn_sisdr_pit_bwd(const float* est, const float* tgt, const int64_t* perm, int B, int S, int T, float eps,
                      const double* fwd_scratch, const float* grad_loss_b, float coef, float* d_est, ctn_stream_t stream);

/* Training-step remainder, egs/wsj0-mix/common/src/driver.py:152-155 (clip_grad_norm_(max_norm) + Adam.step()), on the flat
 * gradient bucket of ctn_convtasnet_bwd: g *= min(1, max_norm/(||g||+1e-6)) (max_norm <= 0: no clipping), then torch.optim.Adam
 * arithmetic (amsgrad off).  params: device array of n_tensors parameter pointers; flat_off / numel: element offset of each
 * tensor's gradient inside flat_grad / its size; exp_avg, exp_avg_sq: Adam state laid out like flat_grad; lr (float) and step
 * (int64, advanced by one) are DEVICE scalars (graph-replayable); chunk_table: int32 pairs (tensor, offset) from
 * ctn_clip_adam_chunks (host helper: returns the chunk count; pass null outputs to size the table); norm_out nullable (1). */
int ctn_clip_adam_chunks(const int* numel, int n_tensors, int* chunk_tensor, int* chunk_offset, int capacity);
int ctn_clip_adam_step(const int32_t* chunk_table, int n_chunks, float* const* params, const long long* flat_off,
                       const int32_t* numel, int n_tensors, const float* flat_grad, size_t flat_numel, float* exp_avg,
                       float* exp_avg_sq, double* sumsq_scratch, const float* lr, long long* step, float beta1, float beta2, float eps,
                       float weight_decay, float max_norm, float* norm_out, ctn_stream_t stream);

/* number of kernel launches the last ctn_* call on this thread enqueued (for bench.py's gpu_launches) */
int ctn_last_launch_count(void);
/* kernels launched by this thread through the library since it was loaded (paths made of several entry calls: DPRNN) */
long long ctn_total_launch_count(void);

/* Stage timing with CUDA events recorded on the launching stream (bench.py's roofline leg).  ctn_profile_enable(1)
 * makes every following ctn_* call on this thread bracket its kernel groups with events; ctn_profile_read
 * synchronises on them, ADDS per-stage milliseconds / launch counts into the caller's arrays (length CTN_NSTAGES)
 * and recycles the events. */
enum ctn_stage {
  CTN_ST_PREP = 0,   /* weight folding / operand images           */
  CTN_ST_ENC = 1,    /* encoder                                   */
  CTN_ST_HEAD = 2,   /* gLN0 + bottleneck 1x1                     */
  CTN_ST_PW1 = 3,    /* per block: 1x1 B->H (+PReLU, stats)       */
  CTN_ST_DW = 4,     /* per block: gLN1 + depthwise + PReLU       */
  CTN_ST_PW2 = 5,    /* per block: [out;skip] 1x1 H->B+Sc         */
  CTN_ST_FIN = 6,    /* per block: residual / skip accumulation   */
  CTN_ST_MASK = 7,   /* PReLU + mask 1x1 + sigmoid + w*mask       */
  CTN_ST_DEC = 8,    /* decoder                                   */
  CTN_ST_LOSS = 9,   /* SI-SDR + PIT                              */
  CTN_NSTAGES = 10
};
int ctn_profile_enable(int enable);
int ctn_profile_read(double* ms, int* launches);

#ifdef __cplusplus
}
#endif
#endif /* CTN_B200_H */
