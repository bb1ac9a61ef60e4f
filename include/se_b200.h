/*
 * se_b200.h -- C-ABI of the B200-native streaming speech-enhancement hot path.
 *
 * Drop-in boundary for the chunked `realtime_process` path of KI-D/Speech-Enhancement-Mi's CRN_ELU.TemporalCRN
 * (and the distilled student of distillation_crn.py).  The reference has no native code: each entry point below
 * replaces a PyTorch call site of the reference, cited as file:line into the reference tree.  No torch types cross
 * this boundary: plain pointers (device pointers unless the name ends in `_host`), sizes and an opaque CUDA stream
 * handle (`void*` = cudaStream_t, NULL = default stream).
 *
 * Every function returns 0 on success and a non-zero status on failure; the message is available from
 * se_last_error() (thread-local).  Nothing throws across the ABI.  There is no CPU fallback: without a CUDA device
 * se_ctx_create fails.
 */
#ifndef SE_B200_H
#define SE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SE_MAX_LEVELS 8

/* numerics variants: CRN_ELU.py (teacher) vs distillation_crn.py:51,340 (student) */
#define SE_VARIANT_CRN_ELU 0
#define SE_VARIANT_DISTILLED 1

/* arithmetic of the dense contractions */
#define SE_PRECISION_FP32 0 /* fp32 FMA on CUDA cores (exact mode)                     */
#define SE_PRECISION_TF32 1 /* tcgen05.mma kind::tf32, fp32 accumulate in TMEM (fast)  */
#define SE_PRECISION_FP16 2 /* tcgen05.mma kind::f16: GEMM operands (activations between layers, weights) stored as
                               fp16 (same 11-bit significand as tf32), fp32 accumulate, fp32 statistics / state / I/O */
#define SE_PRECISION_3XTF32 3 /* tcgen05.mma kind::tf32 on split operands (x = tf32 head + tf32 tail, three products
                                 per step), exact-mode epilogues: fp32-accurate at tensor-core speed */

/* Mirrors the kwargs of CRN_ELU.TemporalCRN.__init__ (CRN_ELU.py:321-323; config.yaml:205-217), with
 * win_length / hop_length already converted from milliseconds to samples (speechbrain STFT: round(sr/1000*ms)). */
typedef struct se_crn_config {
    int32_t num_inputs;                  /* microphones M (3)                              */
    int32_t num_freqs;                   /* F = n_fft/2+1 (201)                            */
    int32_t num_levels;                  /* len(num_channels) (4)                          */
    int32_t num_channels[SE_MAX_LEVELS]; /* [16,32,64,128] teacher / [16,32,64,64] student */
    int32_t hidden;                      /* GRU hidden (512 / 128)                         */
    int32_t num_layers;                  /* GRU layers (2)                                 */
    int32_t kernel_size;                 /* temporal kernel of encoder/decoder (3)         */
    int32_t segment_length;              /* chunk K (3200); hop is K/2                     */
    int32_t n_fft;                       /* 400                                            */
    int32_t win_length;                  /* samples (400)                                  */
    int32_t hop_length;                  /* samples (160)                                  */
    int32_t variant;                     /* SE_VARIANT_*                                   */
    int32_t precision;                   /* SE_PRECISION_*                                 */
    int32_t max_streams;                 /* capacity of the per-stream state arena         */
    int32_t training;                    /* 0: streaming inference context; 1: training context (se_crn_train_*):
                                            max_streams then counts chunk-streams = chunks * utterances per step,
                                            every layer keeps its activations, precision must be FP32 or TF32      */
} se_crn_config;

typedef struct se_ctx se_ctx;

/* ---- lifetime / errors ------------------------------------------------------------------------------------ */
/* replaces: TemporalCRN.__init__ + .to(device)  (CRN_ELU.py:321-365; train.py:58,72; predict.py:45-48) */
int se_ctx_create(se_ctx** out, int device, const se_crn_config* cfg);
int se_ctx_destroy(se_ctx* ctx);
/* thread-local message of the last failing call (the reference raises Python exceptions; SURVEY.md section 8(b)) */
const char* se_last_error(void);
/* library / build identification, e.g. "se_b200 0.1 sm_100a" */
const char* se_version(void);

/* ---- parameters --------------------------------------------------------------------------------------------- */
/* The DISTINCT parameter tensors of TemporalCRN.state_dict() in a fixed order (alias keys `net.0.*` excluded;
 * CRN_ELU.py:225,282).  replaces: nn.Module parameter registration / load_state_dict (train.py:110; predict.py:47). */
int se_crn_num_params(const se_ctx* ctx);
const char* se_crn_param_name(const se_ctx* ctx, int index);
int64_t se_crn_param_numel(const se_ctx* ctx, int index);
/* ptrs[i] -> contiguous fp32 tensor i (device or host memory, reference layout).  The library re-lays the
 * weights out for its kernels; call again after every change of the parameters. */
int se_crn_bind_weights(se_ctx* ctx, const float* const* ptrs, int n, void* stream);

/* ---- per-stream state (CRN_ELU.py:158,228 buffers + GRU h; reset: CRN_ELU.py:408-415) ------------------------ */
/* zero the causal-conv buffers, GRU state and overlap-add carry of streams [first, first+count) */
int se_crn_state_reset(se_ctx* ctx, int first, int count, void* stream);
/* bytes of carried state per stream (SURVEY.md section 8(a) a12): exactly the size of one export record
 * (0 for a training context, which has no streaming state to export) */
int64_t se_crn_state_bytes_per_stream(const se_ctx* ctx);
/* Export / import of the carried state of chosen rows (compaction, migration between contexts or GPUs, checkpoints).
 * A record holds everything the next step of a stream reads (DESIGN.md section 3), se_crn_state_bytes_per_stream bytes,
 * its layout fixed by the model, configuration, precision and front path, never by max_streams or the device.
 *   export: record i of dst_dev <- row rows_host[i] (rows may repeat); the context's state is only read
 *   import: row rows_host[i] <- record i of src_dev (rows must be distinct); `layout` is se_crn_state_layout of the
 *           exporting context and must equal this context's
 * rows_host[i] in [0, max_streams); dst / src are 16-byte aligned device buffers of n records.  Both calls are ordered on
 * `stream` with the steps, do not synchronise the host and keep captured step graphs valid (import writes in place).
 * Training contexts reject both. */
uint64_t se_crn_state_layout(const se_ctx* ctx);
int se_crn_state_export(se_ctx* ctx, const int32_t* rows_host, int n, void* dst_dev, void* stream);
int se_crn_state_import(se_ctx* ctx, const int32_t* rows_host, int n, const void* src_dev, uint64_t layout,
                        void* stream);

/* ---- the fused hot path: one chunk step for B streams --------------------------------------------------------
 * replaces one iteration of the loop CRN_ELU.py:485-489 plus its share of preprocessing/postprocessing
 * (stft_trans :417-424, forward :367-406, istft_trans :426-432, over_add utility.py:393-403).
 *   in  : chunk of K samples per stream and microphone: in[b*in_stream_stride + m*in_mic_stride + n]
 *   out : K/2 samples per stream: (first half of this chunk's iSTFT + carried second half of the previous)/2
 * The carry is always updated.  Streams are rows [0,B) of the state arena.                                      */
int se_crn_process_chunk(se_ctx* ctx, const float* in, int64_t in_stream_stride, int64_t in_mic_stride,
                         float* out, int64_t out_stream_stride, int B, void* stream);

/* replaces: TemporalCRN.realtime_process(mixture[B,M,L], flag) -> [B,L]  (CRN_ELU.py:472-509) on device memory.
 * mixture and out are contiguous [B,M,L] / [B,L].  flag=0 prepends K/2 zeros, resets state and strips the pad.    */
int se_crn_realtime_process(se_ctx* ctx, const float* mixture, int B, int64_t L, int flag, float* out,
                            void* stream);
/* same with HOST buffers: host->device and device->host copies happen inside (this is what predict.py:48,92 times,
 * where model and tensors sit on the CPU). Synchronous. */
int se_crn_realtime_process_host(se_ctx* ctx, const float* mixture, int B, int64_t L, int flag, float* out);

/* ---- the pieces, for callers that use the reference's finer-grained methods ----------------------------------- */
/* replaces: TemporalCRN.stft_trans (CRN_ELU.py:417-424; fullsubnet.py:835-844): chunks [R,M,K] -> spectrum [R,M,F,T,2]
 * (reference layout).  The transforms do not depend on a model: ctx may be NULL (current device). */
int se_stft_trans(se_ctx* ctx, const float* chunks, int R, float* spec, void* stream);
/* replaces: TemporalCRN.istft_trans (CRN_ELU.py:426-432): spectrum [R,F,T,2] -> [R,K] */
int se_istft_trans(se_ctx* ctx, const float* spec, int R, float* out, void* stream);
/* replaces: TemporalCRN.forward (CRN_ELU.py:367-406): x [B,M,F,T,2] -> enhanced spectrum [B,F,T,2]; advances state */
int se_crn_forward_chunk(se_ctx* ctx, const float* spec_in, float* spec_out, int B, void* stream);
/* replaces: utility.segmentation (utility.py:339-370): [B,C,L] -> [B*N,C,K]; *gap / *n_chunks as the reference */
int se_segmentation(const float* x, int B, int C, int64_t L, int K, float* out, int* gap, int* n_chunks,
                    void* stream);
/* chunk-grid arithmetic only (host, no GPU): gap and N for a signal of L samples (utility.py:325-327,357-368) */
int se_chunk_grid(int64_t L, int K, int* gap, int* n_chunks);
/* replaces: utility.over_add (utility.py:373-403): [C,N,K] -> [C, N*K/2 - K/2 - gap] */
int se_over_add(const float* chunks, int C, int N, int K, int gap, float* out, void* stream);

/* ==== FullSubNet (fullsubnet.py:685-961; config.yaml:153-172) ==================================================== */
typedef struct se_fsn_config {
    int32_t num_freqs;        /* 201                                   */
    int32_t num_mics;         /* 3                                     */
    int32_t fb_hidden;        /* fb_model_hidden_size (512)            */
    int32_t sb_hidden;        /* sb_model_hidden_size (384)            */
    int32_t num_layers;       /* 2                                     */
    int32_t sb_num_neighbors; /* 15                                    */
    int32_t fb_num_neighbors; /* 0                                     */
    int32_t max_streams;      /* capacity of the per-stream LSTM state */
    int32_t precision;        /* SE_PRECISION_TF32, SE_PRECISION_3XTF32 (fp32-accurate products and cells), or
                                 SE_PRECISION_FP16: sub-band LSTM operands (98.7 % of the FLOPs) stored as fp16 -- the
                                 reference itself runs this model under fp16 autocast on CUDA (fullsubnet.py:943) */
} se_fsn_config;
typedef struct se_fsn se_fsn;

/* replaces: FullSubNet.__init__ + .cuda() (fullsubnet.py:686-767; predict_fullsubnet.py:31-33) */
int se_fsn_create(se_fsn** out, int device, const se_fsn_config* cfg);
int se_fsn_destroy(se_fsn* ctx);
/* the 20 parameter tensors of FullSubNet.state_dict() (fb_model.*, sb_model.*) in a fixed order */
int se_fsn_num_params(const se_fsn* ctx);
const char* se_fsn_param_name(const se_fsn* ctx, int index);
int64_t se_fsn_param_numel(const se_fsn* ctx, int index);
int se_fsn_bind_weights(se_fsn* ctx, const float* const* ptrs, int n, void* stream);
/* replaces: FullSubNet.reset_state (fullsubnet.py:826-832): zero LSTM states, reset both CumLayerNorms; also zeroes
 * the overlap-add carry of se_fsn_process_chunk */
int se_fsn_reset_state(se_fsn* ctx, int first, int count, void* stream);
/* export / import of the carried state of chosen rows, as se_crn_state_export / se_crn_state_import: both LSTM layers'
 * h and c of the full-band and every sub-band sequence, both CumLayerNorms and the overlap-add carry */
int64_t se_fsn_state_bytes_per_stream(const se_fsn* ctx);
uint64_t se_fsn_state_layout(const se_fsn* ctx);
int se_fsn_state_export(se_fsn* ctx, const int32_t* rows_host, int n, void* dst_dev, void* stream);
int se_fsn_state_import(se_fsn* ctx, const int32_t* rows_host, int n, const void* src_dev, uint64_t layout,
                        void* stream);
/* replaces: FullSubNet.forward on one chunk (fullsubnet.py:769-824), T = 21 frames:
 *   x [B, 2M, F, T] (M real planes then M imaginary planes, fullsubnet.py:835-844) -> compressed cIRM [B, 2, F, T];
 *   advances the LSTM states fh / sh and the CumLayerNorm running means of streams [0, B). */
int se_fsn_forward_chunk(se_fsn* ctx, const float* x, float* out, int B, void* stream);
/* true-streaming FullSubNet step (not in the reference; the chunk loop of fullsubnet.py:932-957 for ONE chunk):
 *   in  : in[b*in_stream_stride + m*in_mic_stride + n], n < 3200, streams = rows [0, B) of the state arena
 *   out : 1600 samples per stream at out[b*out_stream_stride + n] =
 *         (first half of this chunk's iSTFT + carried second half of the previous chunk's) / 2
 * Advances the LSTM states, both CumLayerNorms and the carry of streams [0, B).  No host synchronisation.
 * STFT, network, mask, iSTFT and overlap-add run as one CUDA-graph replay per call (captured once per B). */
int se_fsn_process_chunk(se_fsn* ctx, const float* in, int64_t in_stream_stride, int64_t in_mic_stride,
                         float* out, int64_t out_stream_stride, int B, void* stream);
/* replaces: the layout half of FullSubNet.stft_trans / preprocessing (fullsubnet.py:835-844, 880-886): spectrum
 * [R, M, F, T, 2] (se_stft_trans) -> x [R, 2M, F, T] (M real planes, then M imaginary planes) and / or the mic-0 pair
 * x0 [R, 2, F, T]; either output may be NULL */
int se_fsn_planes(const float* spec, int R, int M, int F, int T, float* x, float* x0, void* stream);
/* replaces: FullSubNet.realtime_process (fullsubnet.py:903-961), everything on the device in one call: front pad (flag = 0),
 * segmentation, per-chunk STFT, the chunk loop (train = 0, :932-945; one CUDA-graph replay per chunk) or all chunks as ONE
 * forward (train = 1, :921-927: both CumLayerNorms see the whole utterance), decompress_cIRM, complex mask, iSTFT and
 * both overlap-adds.  mixture [B, M, L], source [B, M, L] or NULL -> pred [B, L]; optional outputs (NULL to skip):
 * crm [N, B, 2, F, T] (compressed mask), s [N, B, 2, F, T] (mic-0 spectrum of `source`), x0 [N, B, 2, F, T] (mic-0
 * spectrum of the mixture), N = chunks of se_chunk_grid(L + (flag ? 0 : 1600)).  flag = 1 continues the carried state. */
int se_fsn_realtime_process(se_fsn* ctx, const float* mixture, const float* source, int B, int64_t L, int flag, int train,
                            float* pred, float* crm, float* s, float* x0, void* stream);
/* replaces: decompress_cIRM + complex multiply with mic 0 (fullsubnet.py:949-953):
 *   crm [R, 2, F, T], x [R, 2, F, T] (mic-0 real / imaginary) -> enhanced spectrum [R, F, T, 2] */
int se_fsn_apply_mask(const float* crm, const float* x, float* out, int R, int F, int T, void* stream);
/* replaces: BaseModel.unfold (fullsubnet.py:299-331): [B, C, F, T] -> [B, F, C, 2n+1, T], reflect padding (n >= 1),
 * n = 0 is the plain permutation */
int se_unfold(const float* in, int B, int C, int F, int T, int num_neighbor, float* out, void* stream);

/* ==== loss terms of compute_loss, forward only (CRN_ELU.py:513-535; fullsubnet.py:964-987) ======================== */
/* replaces: utility.cal_si_snr (utility.py:207-223): separated, source [B, L] and length [B] (int32, DEVICE memory,
 * may be NULL = full length) -> *out (device scalar) = mean over the batch of the SI-SNR in dB */
int se_cal_si_snr(const float* separated, const float* source, const int32_t* length_dev, int B, int64_t L, float* out,
                  void* stream);
/* replaces: utility.stoi_loss (utility.py:821-916, reduction="mean"): y_true, y_pred [B, L], lens [B] (int32, device)
 * -> *out (device scalar) = -mean(STOI-like score); items whose silent-frame-removed length is <= 512 score 0.99 */
int se_stoi_loss(const float* y_true, const float* y_pred, const int32_t* lens_dev, int B, int64_t L, float* out,
                 void* stream);

/* ==== training micro-step (train.py:195-204; CRN_ELU.py:472-535) =================================================
 * The reference trains through PyTorch autograd: realtime_process (serial chunk loop) -> compute_loss -> backward ->
 * clip_grad_norm_(5) -> Adam.  Here the forward runs batched over all chunks of all utterances (only the GRU
 * recurrence is serial over chunks), every adjoint is a hand-written kernel, and parameters / gradients cross the
 * ABI as ONE flat fp32 vector: the tensors of se_crn_param_name() order, each in the reference layout, concatenated
 * (tensor i starts at se_crn_param_offset(i); se_crn_num_theta() elements in total). */
int64_t se_crn_num_theta(const se_ctx* ctx);
int64_t se_crn_param_offset(const se_ctx* ctx, int index);
/* re-lay the weights out from the flat DEVICE vector (no host round trip; after an optimizer step) */
int se_crn_bind_weights_flat(se_ctx* ctx, const float* theta, void* stream);
/* replaces: model.realtime_process(mixture[B,M,L], flag) in train mode (train.py:195; CRN_ELU.py:472-509):
 * pred [B,L]; keeps what the backward needs.  flag=1 continues the previous piece (state carried, no front pad). */
int se_crn_train_forward(se_ctx* ctx, const float* mixture, int B, int64_t L, int flag, float* pred, void* stream);
/* replaces: the autograd backward from pred to the parameters (train.py:198): dpred [B,L] = d loss / d pred ->
 * grad_flat [num_theta] (overwritten; parameters the graph does not reach, CRN_ELU.py:394-397, get 0) */
int se_crn_train_backward(se_ctx* ctx, const float* dpred, float* grad_flat, void* stream);
/* Distillation feature taps (distillation_crn.py:343-377, 454-470): the student / teacher forward also returns five
 * PRE-activation tensors -- last encoder conv (distillation_crn.py:198,355), GRU Linear (:140,364), and the num_levels-1
 * gated-skip transposed convs (:253,369-371).  se_crn_train_tap reads tap k of the LAST se_crn_train_forward as
 * [chunks*B][C][F][T] (chunk-major rows n*B+i, the reference's torch.cat(f, dim=0) order, distillation_crn.py:466);
 * tap 1 is the Linear output merely re-shaped to (C, F, T) exactly as the reference does.  se_crn_train_backward_taps is
 * se_crn_train_backward with d loss / d tap_k added at the same points (entries may be NULL), i.e. the autograd backward
 * of `loss + distillation_loss(ft, fs)` (distillation_crn.py:560-565) from the student's side. */
int se_crn_train_num_taps(const se_ctx* ctx);
int se_crn_train_tap_shape(const se_ctx* ctx, int tap, int* C, int* F, int* T);
int se_crn_train_tap(se_ctx* ctx, int tap, float* out, void* stream);
int se_crn_train_backward_taps(se_ctx* ctx, const float* dpred, const float* const* dtaps, int n_taps, float* grad_flat,
                               void* stream);
/* se_crn_train_backward_taps, plus d loss / d mixture of the last se_crn_train_forward (the mixture as an autograd input
 * of realtime_process; the carried conv buffers and GRU state are detached as in CRN_ELU.py:185,243, so a sample's
 * gradient comes only from the one or two chunks whose own STFT reads it):
 *   mixture  [B, M, L], the signal that forward read (its 3-mic spectrum is recomputed)
 *   dmixture [B, M, L], overwritten; may be NULL (then this is se_crn_train_backward_taps)
 *   grad_flat may be NULL: parameter-gradient GEMMs are skipped (input gradient only, frozen model) */
int se_crn_train_backward_input(se_ctx* ctx, const float* mixture, const float* dpred, const float* const* dtaps,
                                int n_taps, float* grad_flat, float* dmixture, void* stream);
/* replaces: compute_loss (CRN_ELU.py:513-535) with its backward: source, pred [B,L], length [B] (int32, device) ->
 * out3 (device) = {stoi_loss, cal_si_snr} = {-mean STOI-like score, mean SI-SNR dB} and their gradients w.r.t. pred
 * (d_stoi, d_sisnr: [B,L] each, device).  The caller forms loss = 0.7 * stoi + 0.3 * (-sisnr). */
int se_loss_terms_grad(const float* source, const float* pred, const int32_t* length_dev, int B, int64_t L,
                       float* out2, float* d_stoi, float* d_sisnr, void* stream);
/* out[i] = a * x[i] + b * y[i] with DEVICE scalars *a, *b (combines the two loss gradients with autograd's weights) */
int se_axpby_dev(const float* a, const float* x, const float* b, const float* y, float* out, int64_t n, void* stream);
/* replaces: clip_grad_norm_(params, max_norm) + Adam.step (train.py:200-204; config.yaml:10,99-100) on the flat
 * vectors: *norm_out (device, may be NULL) = total L2 norm before clipping; grad is scaled by
 * min(1, max_norm / (norm + 1e-6)) (max_norm <= 0: no clipping) and `grad_scale` (1 / world size after a summing
 * all-reduce), then theta, m, v are updated in place with bias correction for step `step` (1-based). */
int se_clip_adam_step(float* theta, float* grad, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                      float eps, int step, float max_norm, float grad_scale, float* norm_out, void* stream);

/* ---- introspection used by bench.py --------------------------------------------------------------------------- */
/* number of kernel launches one se_crn_process_chunk issues (graph nodes included) */
int se_crn_launches_per_chunk(const se_ctx* ctx);
/* enable (1) / disable (0) CUDA-graph replay of the chunk step; default 1 */
int se_crn_set_graph(se_ctx* ctx, int enable);
/* time one named stage of the chunk step in isolation: runs it `iters` times on B streams and returns the average
 * device time in milliseconds in *ms.  Stages: "stft", "mask_istft", "step".  Used for the roofline report. */
int se_crn_time_stage(se_ctx* ctx, const char* stage, int B, int iters, float* ms);

/* Kernel-level view of one chunk step, in launch order (the evidence behind bench.py's roofline object):
 * name, algorithmic FLOPs and algorithmic HBM bytes per stream and chunk (SURVEY.md section 8(d)), stage index. */
int se_crn_num_kernels(const se_ctx* ctx);
int se_crn_kernel_info(const se_ctx* ctx, int index, char* name, int name_cap, double* flops_per_stream,
                       double* bytes_per_stream, int* stage);
/* average device time (CUDA events on the launching stream) of kernel `index` alone, launched `iters` times on B streams */
int se_crn_time_kernel(se_ctx* ctx, int index, int B, int iters, float* ms);

/* ---- test hook ------------------------------------------------------------------------------------------------- */
/* Copy the logical interior of a named internal activation of stream b to HOST memory as [T][F][C] (channels-last),
 * dims = {T, F, C}.  Names: "pre_in<i>", "enc_in<i>", "dec_in<j>", "xg", "fcraw", "hseq<l>", "ylast", "noisy".
 * Synchronises the device.  Used by tests/ to localise a parity failure to one layer (CRN_ELU.py:375-399). */
int se_debug_read(se_ctx* ctx, const char* name, int b, float* host_dst, int64_t max_floats, int* dims);
/* Run ONLY the fused mask stage of the chunk step (last GlobalLayerNorm made an identity, decompress_cIRM of
 * utility.py:439-442, complex multiply with the mic-0 spectrum of CRN_ELU.py:401-405) on caller data, all DEVICE memory:
 * mask [B, T, F, 2] (the values that enter decompress_cIRM), noisy [B, T, F, 2] -> spec_out [B, F, T, 2] (the layout
 * forward() returns).  Lets tests drive the clamp |m| >= 9.9, which random-init weights never reach.  Synchronises. */
/* Diagnostic: cycle accounting of the warp roles of the TMA tcgen05 GEMM (contexts created with SE_B200_GEMM_PROFILE=1):
 * out8 = {MMA thread waiting for operands, for a drained accumulator, MMA loop total, producer waiting for a free stage,
 * producer total, epilogue waiting for an accumulator, epilogue total, tiles}, summed over CTAs since the last reset. */
int se_debug_gemm_counters(uint64_t* out8, int reset);
/* Same for the wavefront GRU (builds with -DSE_GRU_PROFILE=1): out16 = [layer][{producer waiting for the published state,
 * producer waiting for a free stage, MMA warp waiting for operands, MMA warp total, epilogue waiting for the accumulator,
 * epilogue total, MMA warp waiting for the drained accumulator, steps}]. */
int se_debug_gru_counters(uint64_t* out16, int reset);
int se_debug_mask_spectrum(se_ctx* ctx, const float* mask, const float* noisy, float* spec_out, int B);

#ifdef __cplusplus
}
#endif
#endif /* SE_B200_H */
