/* libctcb200 — C ABI of the B200-native CTC acoustic hot path.
 *
 * Every entry point takes raw device pointers, sizes and the CUDA stream to enqueue on, returns 0 on
 * success or a negative ctcb200 status, never throws and never allocates memory the caller must free.
 * The message for the last failure on the calling thread is available from ctcb200_last_error().
 * All work is asynchronous on `stream`; nothing here synchronises the device.
 *
 * The reference (Diamondfan/CTC_pytorch) is pure Python on top of PyTorch, so it has no FFI of its own;
 * each function below names the reference call site (file:line under /root/reference) whose library call
 * it replaces. The Python mirror of the reference's classes (ctc_pytorch_b200/*.py) binds these with ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 */
#ifndef CTCB200_H_
#define CTCB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(CTCB200_BUILD)
#define CTCB200_API __attribute__((visibility("default")))
#else
#define CTCB200_API
#endif

/* CUDA stream handle (cudaStream_t) passed as an opaque pointer so this header needs no CUDA include. */
typedef void* ctcb200_stream_t;

enum {
    CTCB200_OK = 0,
    CTCB200_ERR_INVALID = -1,
    CTCB200_ERR_CUDA = -2,
    CTCB200_ERR_DRIVER = -3,
    CTCB200_ERR_TIMEOUT = -4
};

CTCB200_API const char* ctcb200_last_error(void);
CTCB200_API int ctcb200_version(void);

/* ---- CTC loss: replaces nn.CTCLoss(reduction='sum') fwd/bwd, timit/steps/train_ctc.py:144,47,63 ------
 * log_probs [T,N,C] f32; targets [N,*] int64 zero-padded rows of pitch target_stride
 * (timit/utils/data_loader.py:125,140); input_lengths / target_lengths [N] int64.
 * alpha_ws: caller-provided, 16-byte aligned workspace of ctcb200_ctc_workspace_floats(T,N,max_target_len) floats (alpha and
 * beta histories + their log-scale offsets; fwd runs both sweeps concurrently, bwd is the parallel gradient kernel), kept
 * between fwd and bwd. nll [N] f32 = per-utterance negative log likelihood (+inf if infeasible).
 * bwd writes grad [T,N,C] f32 = grad_scale * grad_nll[n] * (exp(lp) - exp(lcab + nll - lp)), zero for
 * t >= input_length (torch's native convention); grad_nll may be NULL (= all ones).
 * Two forms, chosen by the batch size alone (so fwd and bwd of one call pair always agree): below the threshold the latency form
 * above; from N >= threshold the throughput form — fwd runs only the alpha sweeps, bwd runs the beta sweep and emits each frame's
 * gradient row as it goes (no beta history, no separate gradient pass). ctcb200_ctc_set_fused_min_batch sets the threshold
 * (default 2048 — where the two forms cross on a B200 at T = 800 —, or CTCB200_CTC_FUSED_MIN_N at load time; 0 = always, negative = query only) and returns the previous value; it
 * must not change between a fwd and its bwd. */
CTCB200_API int ctcb200_ctc_set_fused_min_batch(int min_batch);
CTCB200_API int64_t ctcb200_ctc_workspace_floats(int T, int N, int max_target_len);
CTCB200_API int ctcb200_ctc_loss_fwd(const float* log_probs, const int64_t* targets, int64_t target_stride,
                                     const int64_t* input_lengths, const int64_t* target_lengths, int T, int N,
                                     int C, int max_target_len, int blank, float* alpha_ws, float* nll,
                                     ctcb200_stream_t stream);
CTCB200_API int ctcb200_ctc_loss_bwd(const float* log_probs, const int64_t* targets, int64_t target_stride,
                                     const int64_t* input_lengths, const int64_t* target_lengths, int T, int N,
                                     int C, int max_target_len, int blank, const float* alpha_ws, const float* nll,
                                     const float* grad_nll, float grad_scale, float* grad, ctcb200_stream_t stream);

/* ---- greedy path: replaces torch.max(out,-1) (train_ctc.py:51), the collapse loop of
 * CTC_Model.compute_wer (timit/models/model_ctc.py:187-202) and GreedyDecoder.decode
 * (timit/utils/ctcDecoder.py:162-166). idx_nt [N,T] int32 frame arg-max (first index on ties);
 * labels_nt [N,T] int32 collapsed labels, label_lengths [N] int32. */
CTCB200_API int ctcb200_argmax(const float* log_probs, int T, int N, int C, int* idx_nt, float* max_nt,
                               ctcb200_stream_t stream);
CTCB200_API int ctcb200_greedy_decode(const float* log_probs, const int64_t* lengths, int T, int N, int C, int blank,
                                      int* idx_nt, int* labels_nt, int* label_lengths, ctcb200_stream_t stream);
/* Batched Levenshtein distance (unit costs) between hypothesis rows a [N, a_stride] int32 of lengths a_len [N] int32 (the
 * labels_nt / label_lengths of ctcb200_greedy_decode) and reference rows b [N, b_stride] int64 of lengths b_len [N] int64
 * (the padded targets of data_loader.py:125,140): the editdistance.eval call of CTC_Model.compute_wer
 * (model_ctc.py:200) and Decoder._edit_distance (ctcDecoder.py:131-149). dist [N] int32. max_b_len <= 1024. */
CTCB200_API int ctcb200_edit_distance(const int32_t* a, int64_t a_stride, const int32_t* a_len, const int64_t* b,
                                      int64_t b_stride, const int64_t* b_len, int N, int max_b_len, int32_t* dist,
                                      ctcb200_stream_t stream);

/* ---- batch assembly on the device (SURVEY.md §8(f) N2): SpeechDataset.__getitem__'s make_context -> skip_feat -> pad to a
 * multiple of n_downsample (timit/utils/data_loader.py:103-110, timit/utils/tools.py:66-86) and create_input's zero padding
 * (data_loader.py:119-140). feat f32 [sum(L_n), F] = the raw utterance features back to back, offsets int64 [N+1] their row
 * offsets. Writes x f32 [N, T_max, F*(left+right+1)] and input_sizes f32 [N] = L''_n / T_max (T_max = max L''_n, computed by
 * the caller from the lengths). pad_labels: labels int64 [sum(S_n)] + offsets -> targets int64 [N, S_max] zero padded and
 * target_sizes int64 [N]. Pure copies: bit-exact. */
CTCB200_API int ctcb200_assemble_features(const float* feat, const int64_t* offsets, int N, int F, int left, int right,
                                          int skip, int n_downsample, int T_max, float* x, float* input_sizes,
                                          ctcb200_stream_t stream);
CTCB200_API int ctcb200_pad_labels(const int64_t* labels, const int64_t* offsets, int N, int S_max, int64_t* targets,
                                   int64_t* target_sizes, ctcb200_stream_t stream);

/* ---- dense GEMM on tcgen05: C[M,N] (+)= A[M,K] * B[N,K]^T, A/B bf16 with K contiguous (pitches lda/ldb in
 * elements, multiples of 8), fp32 accumulate, C f32 (out_bf16=0) or bf16 (1) with pitch ldc.
 * a_koff/b_koff (multiples of 8) shift the K window of each operand (the h_{t-1} shift of dW_hh).
 * tile_n: 0 = auto, else 64/128/256. max_ctas: 0 = persistent over all SMs, > 0 = cap on the CTA count, < 0 = one
 * tile per CTA (for weight-gradient GEMMs that run on a side stream beside the recurrent kernels). Carries the
 * contractions behind nn.LSTM / nn.Linear at timit/models/model_ctc.py:23-26,33,136-139.
 * ctcb200_gemm_preload: loads every tile width of the GEMM kernel on the current device. CUDA loads kernels lazily at their
 * first launch and that load can wait for whatever is running; a GEMM launched for the first time while a kernel that WAITS FOR
 * ITS OUTPUT is resident (the streamed input projection of ctcb200_lstm_fwd_streamed) would never start. The streamed entry
 * point calls it itself; callers that build their own producer/consumer overlap on top of the GEMM should too. */
CTCB200_API int ctcb200_gemm_preload(void);
CTCB200_API int ctcb200_gemm_tn_bf16(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
                                     int M, int N, int K, int a_koff, int b_koff, int out_bf16, int accumulate,
                                     int tile_n, int max_ctas, ctcb200_stream_t stream);
/* Weight-gradient form: C[M,N] (+)= A[a_roff : a_roff+K, 0:M]^T * B[b_roff : b_roff+K, 0:N] — both operands bf16 with the
 * CONTRACTED index as the row index (pitches lda / ldb in elements, multiples of 8), C f32. a_roff / b_roff shift the row
 * window of each operand (any value: the h_{t-1} shift of dW_hh is N rows); rows and columns outside a tensor read as zero.
 * The operands are consumed as the forward pass / ctcb200_lstm_bwd left them (activations [T*N, I], gate gradients [T*N, 8H]):
 * no transposed copies. Carries dW_ih, dW_hh, dW_fc of autograd's nn.LSTM / nn.Linear backward (train_ctc.py:63). */
CTCB200_API int ctcb200_gemm_atb_bf16(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int M, int N,
                                      int K, int a_roff, int b_roff, int accumulate, int tile_n, int max_ctas,
                                      ctcb200_stream_t stream);


/* ---- bidirectional LSTM layer: replaces nn.LSTM(bias=False, bidirectional=True) fwd/bwd time loops,
 * timit/models/model_ctc.py:23-26,33 and the BPTT behind timit/steps/train_ctc.py:63.
 * Operand layouts (all produced by ctcb200_pack_lstm_weights from the torch-layout fp32 parameters
 * weight_ih_l0[4H,I], weight_hh_l0[4H,H] and their *_reverse twins):
 *   wih_p  bf16 [8H, Ipad]  rows (dir, j, unit_local, gate): B operand of Gx = X * wih_p^T
 *   wihT_p bf16 [I, 8H]     B operand of dX = dG * wihT_p^T
 *   whh_p  bf16 [8H, H]     same row order as wih_p; resident A operand of the forward recurrence
 *   whhT_p bf16 [8H, H]     rows (dir, gate, unit), cols = gate-row unit: A operand of the backward recurrence
 * lstm_fwd: gx f32 [T*N, 8H] (= X * wih_p^T), writes hout f32 [T*N, 2H] (fwd | reverse halves), and when
 * c_save / gates_save are non-NULL the cell states f32 [T*N, 2H] and activated gates (4 x fp16 = 8 bytes per
 * element, [T*N, 2H]) that lstm_bwd consumes. scratch: ctcb200_lstm_scratch_bytes(N, H) bytes.
 * lstm_bwd: dhout f32 [T*N, 2H] -> dg bf16 [T*N, 8H] (gate gradients, wih_p column order). When bn_x / bn_coef are
 * non-NULL the layer output feeds a training-mode BatchNorm1d (model_ctc.py:29-32) whose backward is applied on the fly:
 * dhout is then the gradient w.r.t. the normalised tensor, bn_x f32 [T*N, 2H] the layer output itself and
 * bn_coef f32 [3][2H] comes from ctcb200_bn_bwd_coef.
 * batch_tile: 0 = auto, or 16 / 32 batch columns per CTA group. The recurrent entry points take the DEVICE hidden size: a multiple
 * of 128 in [128, 1024], at most 640 in the split-operand mode. Above 640 the kernels exchange h_t / dG_t through global memory
 * with cooperative launches (no streamed projection / gate gradients: ctcb200_lstm_fwd_ctas / _bwd_plan return 0). Any other
 * hidden size H runs at Hp = 128 * ceil(H / 128) with zero padding (ctcb200_pack_lstm_weights_padded): the Hp - H extra units
 * keep h = c = 0 exactly and every activation / gradient buffer uses the Hp layout. */
CTCB200_API int64_t ctcb200_lstm_scratch_bytes(int N, int H);
/* Split-operand ("x3") precision mode — fp32-grade results from bf16 tensor-core products, for parity with the reference's
 * fp32 nn.LSTM arithmetic (model_ctc.py:23-26) to 1e-3 on every gradient: each fp32 operand v is carried as two bf16 tensors,
 * hi = bf16(v) and lo = bf16(v - hi) (`part` = 0 / 1 in the producers below), and a contraction A*B is accumulated in fp32 as
 * A_hi*B_hi + A_hi*B_lo + A_lo*B_hi (three ctcb200_gemm_tn_bf16 launches with accumulate=1, or three tcgen05.mma chains
 * inside the recurrent kernels). Passing the *_lo operands to lstm_fwd / lstm_bwd selects the mode there: gates_save is then
 * 4 x fp32 = 16 bytes per element and lstm_bwd also writes dg_lo. */
/* Other cell types the reference can be configured with (train_ctc.py:20 supported_rnn, model_ctc.py:23): `cell` = 0 nn.LSTM,
 * 1 nn.GRU, 2 nn.RNN(tanh), 3 nn.RNN(relu); `gates` = 4 / 3 / 1 rows of H in the torch weights. All cells share the LSTM's
 * operand layout with four gate slots per unit — GRU uses (r, z, n, -), RNN (g, -, -, -), unused slots carry zero weights —
 * so packing, Gx / dX / dW GEMMs and the exchange are common. GRU: lstm_bwd writes dg (what the input weights see: the n slot
 * holds dn_pre) and dg_rec (what the recurrent weights see: dn_pre * r), the latter feeding dW_hh; c_save holds h_t. */
CTCB200_API int ctcb200_pack_lstm_weights(const float* wih_f, const float* whh_f, const float* wih_r,
                                          const float* whh_r, void* wih_p, void* wihT_p, void* whh_p, void* whhT_p,
                                          int H, int I, int Ipad, int part, int gates, ctcb200_stream_t stream);
/* Zero-padded packing for a torch hidden size H run at the device hidden size Hp >= H (Hp a multiple of 128 for the recurrent
 * kernels): the same layouts at Hp — wih_p [8Hp, Ipad], wihT_p [I_dev, 8Hp], whh_p / whhT_p [8Hp, Hp] — with zero rows for the
 * units >= H and zero recurrent columns for them. The torch input columns come in blocks of i_blk that sit i_blk_p apart on the
 * device (a layer above a padded one: i_blk = H, i_blk_p = Hp; the first layer: i_blk = i_blk_p = I), so
 * I_dev = (I / i_blk) * i_blk_p <= Ipad, and the device columns between the blocks are zero. H = Hp with i_blk = i_blk_p gives
 * exactly ctcb200_pack_lstm_weights. */
CTCB200_API int ctcb200_pack_lstm_weights_padded(const float* wih_f, const float* whh_f, const float* wih_r,
                                                 const float* whh_r, void* wih_p, void* wihT_p, void* whh_p, void* whhT_p,
                                                 int H, int Hp, int I, int i_blk, int i_blk_p, int Ipad, int part, int gates,
                                                 ctcb200_stream_t stream);
CTCB200_API int ctcb200_lstm_fwd(const float* gx, const void* whh_packed, const void* whh_lo_packed, float* hout,
                                 float* c_save, void* gates_save, void* scratch, int T, int N, int H, int batch_tile,
                                 int cell, ctcb200_stream_t stream);
CTCB200_API int ctcb200_lstm_bwd(const float* dhout, const void* whhT_packed, const void* whhT_lo_packed,
                                 const float* c_save, const void* gates_save, void* dg, void* dg_lo, void* dg_rec,
                                 void* dg_rec_lo, void* scratch, int T, int N, int H, int batch_tile, int cell,
                                 const float* bn_x, const float* bn_coef, void* resident_counter, void* resident_event,
                                 ctcb200_stream_t stream);
/* Scheduling aid for overlapping off-critical-path work (weight-gradient GEMMs) with the latency-bound BPTT kernel:
 * resident_event (NULL = off) is a cudaEvent_t (created with timing disabled) attached to the launch as a programmatic event
 * that fires once every block of the BPTT grid has started: cudaStreamWaitEvent on it from another stream is a dependency
 * the CUDA scheduler can see (preferred). The older variant:
 * resident_counter (NULL = off) points at two zero-initialised uint32 words owned by the caller; word 0 is incremented
 * once per lstm_bwd launch as soon as every CTA of that launch is running. ctcb200_stream_wait_geq makes `stream`
 * wait (a driver stream memory operation, no SM is occupied) until *counter >= value, and ctcb200_lstm_bwd_ctas says
 * how many SMs the BPTT launch occupies, i.e. how many a concurrent kernel may take (gemm max_ctas). */
CTCB200_API int ctcb200_lstm_bwd_ctas(int N, int H, int batch_tile);
CTCB200_API int ctcb200_stream_wait_geq(ctcb200_stream_t stream, const void* counter, uint32_t value);
/* Streamed input projection: the forward recurrence of a layer (model_ctc.py:33, nn.LSTM's time loop) starts while most of its
 * input projection Gx = X * W_ih^T (the first half of the same nn.LSTM call) is still being computed on the SMs the
 * latency-bound recurrent kernel leaves idle. Time is cut into chunks of chunk_T >= 2 scan steps; chunk c of a direction holds the
 * rows that direction visits in its scan steps [c*chunk_T, (c+1)*chunk_T) (forward scan: frames t, reverse scan: frames
 * T-1-t). The caller computes chunk 0 of both directions before the launch (stream order), then — on ANOTHER stream, after
 * ctcb200_stream_wait_geq on resident_counter word 0 (incremented once the whole grid is running) and with gemm max_ctas =
 * SM count - ctcb200_lstm_fwd_ctas() — chunk 1, 2, ... each followed by ctcb200_stream_write_value(gx_ready, gx_base + c)
 * (a driver stream memory operation: *gx_ready = value once the preceding work of that stream has completed). The kernel
 * waits for gx_ready - gx_base >= c (wrap-around compare) before it first touches chunk c.
 * ctcb200_lstm_fwd_ctas: SMs the forward launch occupies when it is a single launch with every cluster resident at once
 * (the only form that can be streamed), else 0 — ask before using ctcb200_lstm_fwd_streamed.
 * ctcb200_concurrency_probe: the streamed form is only legal where a kernel on one stream makes progress while a kernel on
 * another stream is resident. Profilers (Nsight Compute serialises all kernels), CUDA_LAUNCH_BLOCKING and some debug / MPS
 * set-ups do not provide that — the recurrent kernel would wait for chunks that cannot be produced until its timeout trap. The
 * probe runs the pattern in miniature (a one-thread kernel on stream_a polls a flag for at most limit_ms; a trivial kernel and a
 * stream memory operation on stream_b raise it) and returns 1 / 0 (negative: error); it synchronises both streams — call it
 * once per device before choosing the streamed form, and keep the whole-projection form (ctcb200_lstm_fwd) otherwise. */
CTCB200_API int ctcb200_concurrency_probe(ctcb200_stream_t stream_a, ctcb200_stream_t stream_b, int limit_ms);
CTCB200_API int ctcb200_lstm_fwd_streamed(const float* gx, const void* whh_packed, const void* whh_lo_packed, float* hout,
                                          float* c_save, void* gates_save, void* scratch, int T, int N, int H, int batch_tile,
                                          int cell, void* resident_counter, const void* gx_ready, uint32_t gx_base,
                                          int chunk_T, ctcb200_stream_t stream);
CTCB200_API int ctcb200_lstm_fwd_ctas(int N, int H, int batch_tile, int x3, int cell);
CTCB200_API int ctcb200_stream_write_value(ctcb200_stream_t stream, void* counter, uint32_t value);
/* Streamed gate gradients: the mirror image for the backward pass (train_ctc.py:63). lstm_bwd_streamed is lstm_bwd plus a
 * progress counter: every CTA of the launch adds 1 to *progress_counter each time its dG rows of another chunk_T scan steps
 * are written (chunk c = scan steps [c*chunk_T, (c+1)*chunk_T): rows of frames T-1-s for the forward direction's BPTT, frames
 * s for the reverse direction's; the last chunk may be shorter and is counted too). A second stream waits
 * (ctcb200_stream_wait_geq) for base + (c+1) * ctcb200_lstm_bwd_plan() and runs the chunk's share of the input-gradient GEMM
 * dX = dG * W_ih (and, for the first layer, of the weight-gradient contractions) on the SMs the BPTT kernel leaves idle, so
 * that only the last chunk is left when the recurrence ends. ctcb200_lstm_bwd_plan: CTAs of the BPTT launch when it is one
 * clustered launch (the only form that can be streamed), else 0. */
CTCB200_API int ctcb200_lstm_bwd_streamed(const float* dhout, const void* whhT_packed, const void* whhT_lo_packed,
                                          const float* c_save, const void* gates_save, void* dg, void* dg_lo, void* dg_rec,
                                          void* dg_rec_lo, void* scratch, int T, int N, int H, int batch_tile, int cell,
                                          const float* bn_x, const float* bn_coef, void* resident_counter,
                                          void* progress_counter, int chunk_T, ctcb200_stream_t stream);
CTCB200_API int ctcb200_lstm_bwd_plan(int N, int H, int batch_tile, int x3, int cell);

/* ---- layout / normalisation kernels around the GEMMs (model_ctc.py:29-32 BatchNorm1d over T*N rows,
 * model_ctc.py:136-140,165-168 fc BatchNorm + LogSoftmax, model_ctc.py:175 the (N,T,F)->(T,N,F) transpose).
 * cast_transpose: src f32 element (r,c) at src[(r / n_inner)*s_outer + (r % n_inner)*s_inner + c], optional
 * per-column affine v*scale[c]+shift[c]; writes bf16 dst [R, dst_pitch] and/or bf16 dstT [C, dstT_pitch], where
 * the transposed column of row r is (r / n_inner)*n_pad + (r % n_inner): the batch axis is padded to n_pad
 * (a multiple of 8) so that the one-time-step shift of the dW_hh contraction stays 16-byte aligned for TMA.
 * Pad columns are not written; the caller zero-fills dstT when n_pad != n_inner. part = 0: bf16(v); part = 1: the
 * split-operand remainder bf16(v - bf16(v)). */
CTCB200_API int ctcb200_cast_transpose(const float* src, int64_t s_outer, int64_t s_inner, int n_inner,
                                       const float* scale, const float* shift, void* dst, int64_t dst_pitch,
                                       void* dstT, int64_t dstT_pitch, int n_pad, int R, int C, int part,
                                       ctcb200_stream_t stream);

/* ws: 2*C doubles. Batch statistics over R rows of x f32 [R, C]; mean/rstd saved for backward, scale/shift =
 * the affine to apply (gamma*rstd, beta - mean*gamma*rstd); running stats updated with `momentum`
 * (unbiased variance), pass NULL to skip. */
CTCB200_API int ctcb200_bn_train_stats(const float* x, int R, int C, const float* gamma, const float* beta,
                                       float* running_mean, float* running_var, float momentum, float eps,
                                       float* mean, float* rstd, float* scale, float* shift, void* ws, int n_valid,
                                       ctcb200_stream_t stream);
CTCB200_API int ctcb200_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean,
                                       const float* running_var, float eps, float* scale, float* shift, int C,
                                       ctcb200_stream_t stream);
/* dx may alias dy. dgamma / dbeta may be NULL. */
CTCB200_API int ctcb200_bn_bwd(const float* dy, const float* x, const float* mean, const float* rstd,
                               const float* gamma, float* dx, float* dgamma, float* dbeta, int R, int C, void* ws,
                               int n_valid, ctcb200_stream_t stream);
/* Same reduction, but instead of writing dx it emits coef f32 [3][C] with dx = coef[0][c]*dy + coef[1][c]*x + coef[2][c];
 * ctcb200_lstm_bwd applies it while it reads its incoming gradient (bn_x / bn_coef), which saves one pass over [R, C]. */
CTCB200_API int ctcb200_bn_bwd_coef(const float* dy, const float* x, const float* mean, const float* rstd,
                                    const float* gamma, float* coef, float* dgamma, float* dbeta, int R, int C, void* ws,
                                    int n_valid, ctcb200_stream_t stream);
CTCB200_API int ctcb200_log_softmax_fwd(const float* x, int64_t x_pitch, float* y, int R, int C,
                                        ctcb200_stream_t stream);
CTCB200_API int ctcb200_log_softmax_bwd(const float* g, const float* y, float* dx, int R, int C,
                                        ctcb200_stream_t stream);
/* Packed (variable-length) sequences, my_863_corpus/steps/model.py:37-56,93-141 fed by pack_padded_sequence
 * (lstm_ctc.py:41): the recurrent kernels always scan all T rows, so packed semantics come from alignment — the forward
 * direction runs on the left-aligned batch, the reverse direction on a right-aligned copy — plus BatchNorm sums divided by the
 * valid-frame count (n_valid above; 0 = all R rows; padding rows must be zero). realign_rows moves [T,N,W] f32 rows between the
 * two alignments and zeroes the padding: columns [0,split) are masked only (dst = t < len ? src : 0), columns [split,W) are
 * shifted by T-len_n (dir=+1: right->left aligned, dir=-1: left->right aligned); accumulate=1 adds into dst. lengths: i64 [N]. */
CTCB200_API int ctcb200_realign_rows(const float* src, float* dst, const void* lengths_i64, int T, int N, int W, int split,
                                     int dir, int accumulate, ctcb200_stream_t stream);
/* a[e] = mask[e] ? a[e] * inv_keep : 0 (nn.Dropout, model_ctc.py:26,34); mask bytes come from the caller's RNG */
CTCB200_API int ctcb200_dropout_apply(float* a, const void* mask_u8, float inv_keep, int64_t n,
                                      ctcb200_stream_t stream);

/* ---- CNN front: LayerCNN = Conv2d(bias) -> BatchNorm2d -> ReLU (timit/models/model_ctc.py:38-68,148), direct fp32
 * convolution kernels (the front is 0.5 % of the model's FLOPs and too thin for tensor-core tiles). Activations are
 * channel-last [N,H,W,C] f32 between blocks; w / dw are torch's [Cout,Cin,kh,kw] f32; y / dy are rows [M=N*Ho*Wo, Cout].
 * conv2d_fwd: y = conv(x, w) + bias (bias may be NULL). conv2d_wgrad: dw = sum_m dy[m,:] (x) patch(m); ws holds
 * ctcb200_conv2d_wgrad_ws_bytes() bytes of per-CTA partial sums (reduced in a fixed order: deterministic).
 * conv2d_dgrad: dx = conv^T(dy, w), every element written once.
 * affine_act: a(n,h,w,c) = act(y[m,c]*scale[c]+shift[c]) written with strides (sn,sh,sw,sc); scale may be NULL; act = 0 relu,
 * 1 tanh, 2 sigmoid (train_ctc.py:21 supported_activate), 3 identity (layout change only).
 * act_bwd_gather: dz[m,c] = act'(a(n,h,w,c)) * da(n,h,w,c), the derivative taken from the activation's output a.
 * col_sum: out[c] = sum_m y[m,c] (bias gradient). */
CTCB200_API int ctcb200_conv2d_fwd(const float* x_nhwc, const float* w, const float* bias, float* y, int N, int Hi, int Wi,
                                   int Cin, int Cout, int Ho, int Wo, int kh, int kw, int sh, int sw, int ph, int pw,
                                   ctcb200_stream_t stream);
CTCB200_API int64_t ctcb200_conv2d_wgrad_ws_bytes(int Cin, int Cout, int kh, int kw);
CTCB200_API int ctcb200_conv2d_wgrad(const float* x_nhwc, const float* dy, float* dw, void* ws, int N, int Hi, int Wi, int Cin,
                                     int Cout, int Ho, int Wo, int kh, int kw, int sh, int sw, int ph, int pw,
                                     ctcb200_stream_t stream);
CTCB200_API int ctcb200_conv2d_dgrad(const float* dy, const float* w, float* dx_nhwc, int N, int Hi, int Wi, int Cin, int Cout,
                                     int Ho, int Wo, int kh, int kw, int sh, int sw, int ph, int pw,
                                     ctcb200_stream_t stream);
CTCB200_API int ctcb200_add_bias_rows(float* y, const float* bias, int64_t R, int C, ctcb200_stream_t stream);
CTCB200_API int ctcb200_affine_act(const float* y, const float* scale, const float* shift, float* a, int64_t sn,
                                   int64_t sh, int64_t sw, int64_t sc, int N, int Ho, int Wo, int C, int act,
                                   ctcb200_stream_t stream);
CTCB200_API int ctcb200_act_bwd_gather(const float* da, const float* a, float* dz, int64_t sn, int64_t sh, int64_t sw,
                                       int64_t sc, int N, int Ho, int Wo, int C, int act, ctcb200_stream_t stream);
/* nn.MaxPool2d(pool) of LayerCNN (model_ctc.py:53-54,65-66): kernel = stride = pool, floor mode, channel-last tensors;
 * idx_u8 [N,H/kh,W/kw,C] keeps the arg-max position inside each window for the backward pass. */
CTCB200_API int ctcb200_maxpool2d_fwd(const float* x_nhwc, float* y_nhwc, void* idx_u8, int N, int H, int W, int C, int kh,
                                      int kw, ctcb200_stream_t stream);
CTCB200_API int ctcb200_maxpool2d_bwd(const float* dy_nhwc, const void* idx_u8, float* dx_nhwc, int N, int H, int W, int C,
                                      int kh, int kw, ctcb200_stream_t stream);
CTCB200_API int ctcb200_col_sum(const float* y, float* out, int64_t R, int C, ctcb200_stream_t stream);

/* ---- beam decode: replaces ctcBeamSearch.decode, timit/utils/BeamSearch.py:73-153 (called by
 * BeamDecoder.decode, timit/utils/ctcDecoder.py:181-192) with LanguageModel.get_bi_prob
 * (timit/utils/NgramLM.py:65-78) flattened into lm_table f64 [(C+1),(C+1)] (row = previous unit, row C =
 * sentence start; column C = sentence end; NaN = pair unknown to the LM).
 * probs_ntc f32 [N,T,C] are probabilities (ctcb200_exp_transpose produces them from [T,N,C] log-probs like
 * ctcDecoder.py:189-190). Outputs: out_labels int32 [N,T] + out_lengths [N]; status [N]: 0 ok, 1 = the
 * reference would raise IndexError (empty prefix reaches the final LM step), 2 = ValueError (log of a zero
 * probability), 3 = KeyError (unit missing from the LM). workspace: ctcb200_beam_workspace_bytes(...) bytes. */
CTCB200_API int64_t ctcb200_beam_workspace_bytes(int T, int N, int C, int beam_width);
CTCB200_API int ctcb200_exp_transpose(const float* log_probs_tnc, float* probs_ntc, int T, int N, int C,
                                      ctcb200_stream_t stream);
CTCB200_API int ctcb200_beam_search(const float* probs_ntc, const int64_t* lengths, const double* lm_table,
                                    double lm_alpha, int T, int N, int C, int beam_width, int blank, void* workspace,
                                    int* out_labels, int* out_lengths, int* status, ctcb200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CTCB200_H_ */
