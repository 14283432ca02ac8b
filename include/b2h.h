/* b2h.h -- C-ABI of libb2h.so: the B200 (sm_100a) hot path of body2hand.
 *
 * The reference (benoriol/hand_pose_sl) has no FFI of its own: its hot path sits behind the PyTorch
 * Python API.  Each entry point below replaces the work one reference call does and cites it
 * (paths relative to the reference root).  All pointers are DEVICE pointers owned by the caller
 * (torch allocator) unless the name ends in _host; kernels are enqueued on `stream` (a cudaStream_t
 * passed as void*), never allocate, never synchronise, never free -> CUDA-graph capturable.
 * Return value: 0 on success, negative B2H_E* otherwise; b2h_last_error() holds a message
 * (thread-local).  Nothing here throws or exits.
 */
#ifndef B2H_H_
#define B2H_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2H_OK        0
#define B2H_EINVAL   -1   /* null pointer / bad enum */
#define B2H_ESHAPE   -2   /* unsupported shape (C, T, channel count) */
#define B2H_EALIGN   -3   /* pointer not aligned as required */
#define B2H_EARCH    -4   /* device is not sm_100 */
#define B2H_ECUDA    -5   /* CUDA launch error (cudaGetLastError after enqueue) */
#define B2H_EWORKSPACE -6 /* workspace too small */

/* precision modes (north_star: fp32 mode 1e-4, bf16 mode 2e-2) */
#define B2H_FP32 0        /* fp32 mode: tcgen05 with every operand split into bf16 high + low halves, three MMAs per
                             product (x_hi*w_hi + x_lo*w_hi + x_hi*w_lo), fp32 accumulate in TMEM: ~6e-6 relative on the
                             prediction (conv_channels <= 32, T <= 256; windows longer than 128 frames train as overlapping
                             128-frame sub-windows with real context at the cuts); the FFMA kernel for every other shape */
#define B2H_BF16 1        /* tcgen05 kind::f16 (bf16 operands), fp32 accumulate (TMEM) */
#define B2H_FP32_FFMA 2   /* fp32 mode on the CUDA cores only (FFMA, fp32 accumulate): the arbiter of the split kernel */

/* loss kinds -- only the two the reference actually computes (steps/traintest.py:114-117) */
#define B2H_LOSS_L1     0 /* maskedPoseL1     steps/utils.py:413-428 (batch mean) */
#define B2H_LOSS_CONFL1 1 /* poderatedPoseL1  steps/utils.py:431-452 (batch SUM)  */

/* pad rule of a cropped window */
#define B2H_PAD_REPEAT_FIRST 0  /* dataloaders/text_pose_dataset.py:511-518 (JSON datasets) */
#define B2H_PAD_ZEROS        1  /* dataloaders/text_pose_dataset.py:614-622 (H5 dataset)    */

/* element types of activation tensors crossing the ABI */
#define B2H_DT_F32  0
#define B2H_DT_BF16 1

const char* b2h_last_error(void);
int b2h_version(void);
/* 1 if the current device is compute capability 10.x, else 0 (no CPU fallback exists). */
int b2h_device_ok(void);

/* ---- model geometry ------------------------------------------------------------------------
 * ConvModel.__init__  body2hand/src/models/HandPoseModels.py:18-37:
 * conv1 (C, n_in[+1 if pos_emb], 5), conv2/3 (C, C, 5), conv4 (42, C, 5) + biases; the flat fp32
 * parameter buffer holds them in state_dict order conv1.weight, conv1.bias, ..., conv4.bias.
 * `pos_emb` everywhere in this ABI: 0 = off; 1 = LinearPositionalEmbedding with the reference's max_len = 100 (row t/100,
 * models/HandPoseModels.py:23, 66-84); n > 1 = the same row with max_len = n (SURVEY 8f N4: windows other than 100 frames --
 * the reference's torch.cat only works for T == max_len, the kernels generate t/max_len for any T). */
int64_t b2h_param_count(int n_in, int C, int pos_emb);
/* float offset of conv{layer}.weight (is_bias=0) / .bias (is_bias=1) in the flat buffer, layer 1..4 */
int64_t b2h_param_offset(int n_in, int C, int pos_emb, int layer, int is_bias);
/* bytes of the extension-owned packed weight buffer (fp32 tap-major + bf16 UMMA operand layouts) */
int64_t b2h_packed_bytes(int n_in, int C, int pos_emb);
/* Host-only self-check of the internal gradient-partial slot layout of the tensor-core train kernel (flat parameter
 * index <-> slot bijection, padding slots, float4 alignment); returns the number of violations, 0 = consistent. */
int64_t b2h_gp_layout_check(int n_in, int C, int pos_emb);
/* Host-only query of the training path's window decomposition: returns the number of sub-windows a window of T frames is
 * processed as (1 = whole windows; windows longer than a tile segment -- 128 frames in fp32 mode, 256 in bf16 mode -- are cut
 * into overlapping sub-windows of that length that read real context frames at the cuts and apply the criterion to their
 * core rows; T <= 4096) and, when out4 is non-NULL, sub-window i as
 * {first frame, first core row, end of core rows, sub-window length}.  tests/test_tiling_model.py proves the identity
 * "sum of the sub-windows' gradients == the window's gradient" for this decomposition on the CPU. */
int b2h_train_subwindows(int T, int n_in, int C, int pos_emb, int precision, int i, int* out4);

/* bytes of scratch the train entry points need (1-KB header of the fused kernel's grid barrier + per-CTA gradient
 * partials for a deterministic two-stage reduction + loss partials); 16-byte aligned, zeroed once at allocation */
int64_t b2h_workspace_bytes(int B, int T, int n_in, int C, int pos_emb, int precision);
/* 1 if (T, C) is supported by the given precision's kernels (forward AND training) on this build, else 0.  A bf16-mode
 * shape counts as supported when its training runs on the FFMA kernel (see B2H_KERNEL_FFMA). */
int b2h_supported(int T, int n_in, int C, int pos_emb, int precision);
/* 1 if b2h_conv_forward alone covers (T, C) in the given precision -- wider than b2h_supported: bf16 inference runs
 * conv_channels up to 256 (streamed-weight tensor-core kernel) -- else 0 */
int b2h_forward_supported(int T, int n_in, int C, int pos_emb, int precision);
/* Which kernel the forward (train = 0) or the train step (train = 1) runs for this shape -- the dispatch itself uses
 * this function, so a test can pin "the tensor-core path is the one that runs" without a GPU. */
#define B2H_KERNEL_NONE 0        /* unsupported: the entry point returns B2H_ESHAPE */
#define B2H_KERNEL_FFMA 1        /* fp32-accumulate FFMA kernel (B2H_FP32_FFMA; B2H_FP32 beyond the tile kernel; and B2H_BF16
                                    TRAINING where no tensor-core training kernel fits but FFMA's shared memory does: 16 input
                                    channels, no pos_emb, C = 33..36, T = 257..264 -- those steps run with unrounded fp32
                                    operands) */
#define B2H_KERNEL_TC_TILE 2     /* tcgen05 tile kernel, weights resident in shared memory (bf16: C <= 64 fwd / 32 train;
                                    fp32 mode = bf16 high/low pairs: C <= 32; T <= 256) */
#define B2H_KERNEL_TC_ROWSPACE 3 /* tcgen05 layer-major row-space forward (C <= 32 up to T = 1024, C <= 48 up to T = 640,
                                    with up to 32 input channels; at any batch) */
#define B2H_KERNEL_TC_WIDE 4     /* tcgen05 streamed-weight forward (C <= 256, T <= 256) */
#define B2H_KERNEL_TC_WIDE_TRAIN 5 /* tcgen05 wide training (32 < C <= 256, T <= 256, bf16 mode): streamed-weight forward that
                                    saves the layer inputs + criterion, dgrad chain with the transposed blocks, split-K
                                    weight-gradient GEMMs over the saved operands (three launches + reduce/Adam) */
int b2h_kernel_choice(int T, int n_in, int C, int pos_emb, int precision, int train);

/* Re-layout the flat fp32 parameters into the packed buffer (run after load_state_dict / any
 * out-of-band weight change; the fused Adam keeps it fresh by itself). */
int b2h_pack_weights(const float* params, void* packed, int n_in, int C, int pos_emb, void* stream);

/* ---- K0 preprocessing -----------------------------------------------------------------------
 * Replaces, per window slot: load_keypoints + BODY_HEAD_KEYPOINTS gather
 * (dataloaders/text_pose_dataset.py:14-50), crop/pad/clip (…:52-68, 511-529), .float() (…:536-544),
 * WristDifference / ChestDifference / NormalizeFixedFactor / BuildRightHandItem
 * (steps/utils.py:180-210, 261-277).  Bit-exact (IEEE sub.rn then div.rn).
 * Inputs: OpenPose rows [x,y,c]: pose25 (F,25,3), hand_left (F,21,3), hand_right (F,21,3) fp32.
 * Window w covers source frames [win_start[w], win_start[w]+T) cut at win_end[w] (nullable: F) -- the end of the
 * utterance it is cropped from when several utterances are packed back to back -- and padded by `pad_mode`.
 * Outputs (W,T,12,2) (W,T,12) (W,T,21,2) (W,T,21) [(W,T,21,2) (W,T,21)] fp32, every one nullable (an inference stream
 * needs only the keypoint input: at least one output or input_kp_bf16 must be given),
 * n_frames_out (W) int64 = min(F - start, T)  (…:447);  input_kp_bf16 nullable (W,T,24) bf16 copy
 * feeding the bf16 net without a second pass. */
int b2h_preprocess(const float* pose25, const float* hand_left, const float* hand_right, int64_t n_frames,
                   const int64_t* win_start, const int64_t* win_end, int n_win, int T, int pad_mode, float factor, int dif_encoding,
                   int normalize, float* input_kp, float* input_conf, float* target_kp, float* target_conf,
                   float* left_kp, float* left_conf, int64_t* n_frames_out, void* input_kp_bf16, void* stream);

/* 0 = clean, 1 = a preprocessing launch gave up waiting for a staged frame group (bounded spin, ~2 s): its outputs are
 * incomplete.  Reading clears it.  Synchronises the device. */
int b2h_preprocess_status(void);

/* Test aid for the kernel's division: counts, over ALL 2^32 float bit patterns x, the cases where the
 * reciprocal+FMA division used for `factor` differs from IEEE div.rn(x, factor) (must be 0; mismatches_dev is a
 * zero-initialised device uint64). */
int b2h_verify_fastdiv(float factor, unsigned long long* mismatches_dev, void* stream);

/* Same for the packed H5 row format of TextPoseH5Dataset.array2item
 * (dataloaders/text_pose_dataset.py:587-612): rows (F,150) = [x0..x49 | y0..y49 | c0..c49],
 * body = columns 0..7 (8 keypoints), left hand 8..28, right hand 29..49.  Outputs (W,T,8,2) (W,T,8) ... */
int b2h_preprocess_h5(const float* rows150, int64_t n_frames, const int64_t* win_start, const int64_t* win_end, int n_win, int T,
                      int pad_mode, float factor, int dif_encoding, int normalize, float* input_kp,
                      float* input_conf, float* target_kp, float* target_conf, float* left_kp, float* left_conf,
                      int64_t* n_frames_out, void* stream);

/* ---- K1 forward -----------------------------------------------------------------------------
 * ConvModel.forward  models/HandPoseModels.py:40-64 (+ LinearPositionalEmbedding :66-84 when
 * pos_emb).  x (B,T,n_in) NWC [== the reference's (B,T,12,2)], x_dtype fp32 or bf16;
 * y (B,T,42) fp32 [== (B,T,21,2)].  lengths nullable int32 (B): when apply_mask, rows t>=len are
 * written as 0 (mask_output, steps/utils.py:309-312).  out_scale multiplies the result
 * (1280 = the de-normalise of steps/traintest.py:270-271; 1 = none). */
int b2h_conv_forward(const void* x, int x_dtype, const float* params, const void* packed, const int32_t* lengths,
                     float* y, int B, int T, int n_in, int C, int pos_emb, int precision, int apply_mask,
                     float out_scale, void* stream);

/* ConvModel.forward over WINDOW VIEWS of a per-frame stream (BASELINE config 5: sliding windows over hours of frames).
 * frames (n_frames, n_in) fp32 or bf16 = the preprocessed keypoints of every unique frame (b2h_preprocess with ONE window
 * covering the clip); window w, frame t reads row win_start[w] + t, cut at win_end[w] (nullable: n_frames) and padded by
 * `pad_mode` exactly like b2h_preprocess pads a crop (dataloaders/text_pose_dataset.py:52-68, 511-518, 614-622) -- the
 * same result as materialising the (n_win, T, n_in) windows first, without writing or re-reading them (stride 16 = 4x
 * overlap).  y (n_win, T, 42) fp32.  Served by the tensor-core kernels b2h_conv_forward runs: bf16 mode with
 * conv_channels <= 256 and T <= 256, conv_channels <= 48 and T <= 640 or conv_channels <= 32 and T <= 1024 (the last two
 * with up to 32 input channels), fp32 mode with conv_channels <= 32 and T <= 256, at any n_win (B2H_ESHAPE otherwise,
 * including every shape b2h_conv_forward runs on the FFMA kernel). */
int b2h_conv_forward_windows(const void* frames, int x_dtype, int64_t n_frames, const int64_t* win_start, const int64_t* win_end,
                             int pad_mode, const float* params, const void* packed, const int32_t* lengths, float* y, int n_win,
                             int T, int n_in, int C, int pos_emb, int precision, int apply_mask, float out_scale, void* stream);

/* LinearPositionalEmbedding.forward as a stand-alone call (models/HandPoseModels.py:78-84): inp (B, channels, T) fp32
 * -> out (B, channels+1, T) with out[:,0,t] = t / max_len (fp32 division) and the input channels behind it.  Like the
 * reference's torch.cat it only works for T == max_len (B2H_ESHAPE otherwise).  ConvModel(pos_emb=True) does not
 * call this: its kernels generate the row on the fly. */
int b2h_pos_emb_concat(const float* inp, float* out, int B, int channels, int T, int max_len, void* stream);

/* ---- K2 fused forward + loss + backward --------------------------------------------------------
 * One iteration of steps/traintest.py:94-120 up to loss.backward():  forward, mask_output,
 * maskedPoseL1 / poderatedPoseL1, and every parameter gradient (conv dgrad/wgrad/bias-grad, ReLU
 * mask).  grads_out: flat fp32 (b2h_param_count), overwritten; NULL = run only the fused kernel and
 * leave the per-CTA partials in the workspace (per-kernel timing).  loss_out: 1 float.
 * pred_out nullable (B,T,42) masked prediction.  conf (B,T,21) only for B2H_LOSS_CONFL1.
 * step_dev nullable: device int64 step counter, incremented here (see b2h_adam_step / b2h_train_step). */
int b2h_train_forward_backward(const void* x, int x_dtype, const float* target, const float* conf,
                               const int32_t* lengths, const float* params, const void* packed,
                               float* grads_out, float* loss_out, float* pred_out, int B, int T, int n_in, int C,
                               int pos_emb, int loss_kind, int precision, int64_t* step_dev, void* workspace,
                               int64_t workspace_bytes, void* stream);

/* b2h_train_forward_backward over WINDOW VIEWS of device-resident frame streams: training from a preprocessed set kept in
 * device memory, where a step needs only its crop list (win_start, win_end, lengths: 20 B per window) instead of a
 * materialised (n_win, T, .) batch.  frames (n_frames, n_in) fp32 or bf16 (16-byte aligned), target_frames
 * (n_frames, 42) fp32 (8-byte aligned), conf_frames (n_frames, 21) fp32 (4-byte aligned, B2H_LOSS_CONFL1 only): window w,
 * frame t reads the SAME row of all three streams, the crop [win_start[w], win_start[w] + T) cut at min(win_end[w],
 * n_frames) (win_end nullable) and padded by `pad_mode` exactly like b2h_preprocess; a padded row of B2H_PAD_ZEROS is a
 * zero row in all three.  lengths (n_win) as in the dense call (the reference takes them from the metadata, not the
 * crop); pred_out stays dense (n_win, T, 42).  Bit-identical to b2h_train_forward_backward on the windows b2h_preprocess
 * materialises.  Workspace: b2h_workspace_bytes(n_win, T, ...).  Served where b2h_kernel_choice(T, ..., train = 1) is
 * B2H_KERNEL_TC_TILE or B2H_KERNEL_TC_WIDE_TRAIN; B2H_ESHAPE on every FFMA shape. */
int b2h_train_forward_backward_windows(const void* frames, int x_dtype, const float* target_frames, const float* conf_frames,
                                       int64_t n_frames, const int64_t* win_start, const int64_t* win_end, int pad_mode,
                                       const int32_t* lengths, const float* params, const void* packed, float* grads_out,
                                       float* loss_out, float* pred_out, int n_win, int T, int n_in, int C, int pos_emb,
                                       int loss_kind, int precision, int64_t* step_dev, void* workspace,
                                       int64_t workspace_bytes, void* stream);

/* Backward of ConvModel.forward alone for the modular autograd path (what loss.backward() does
 * below the criterion, steps/traintest.py:120): d_y (B,T,42) fp32 -> flat parameter gradients
 * (activations are recomputed in shared memory, nothing was saved by the forward). */
int b2h_conv_backward(const void* x, int x_dtype, const float* d_y, const float* params, const void* packed,
                      float* grads_out, int B, int T, int n_in, int C, int pos_emb, int precision,
                      void* workspace, int64_t workspace_bytes, void* stream);

/* ---- criteria as stand-alone calls (modular API) ------------------------------------------------
 * mask_output  steps/utils.py:309-312 (in place). */
int b2h_mask_output(float* y, const int32_t* lengths, int B, int T, int row_elems, void* stream);
/* maskedPoseL1 / poderatedPoseL1 forward value and d(loss)/d(pred) in one pass
 * (steps/utils.py:413-452).  pred/target (B,T,row_elems), scores (B,T,row_elems/2) nullable,
 * loss_out 1 float, d_pred nullable (B,T,row_elems), row_scratch (B) floats. */
int b2h_pose_l1(const float* pred, const float* target, const float* scores, const int32_t* lengths, int B,
                int T, int row_elems, int loss_kind, float* loss_out, float* d_pred, float* row_scratch,
                void* stream);

/* Inference output formats (after the fused de-normalise of b2h_conv_forward): pred (rows,42) -> out (rows,63).
 * mode 0 = OpenPose hand rows [x,y,1.0]*21 (array2open_pose, steps/utils.py:355-364);
 * mode 1 = packed H5 rows [x*21 | y*21 | 0*21] (order_and_reshape_toh5, steps/traintest.py:302-317). */
int b2h_format_prediction(const float* pred, float* out, int64_t rows, int mode, void* stream);

/* ---- K3 fused Adam ------------------------------------------------------------------------------
 * torch.optim.Adam.step with torch defaults (steps/traintest.py:48,121) over the flat buffer:
 * g = grads*grad_scale (grad_scale = 1/world for data parallel); m,v,p updated in place; when
 * `packed` is non-null the new weights are also scattered into the packed operand layouts so the
 * next forward needs no re-pack.  step is 1-based; step_dev (nullable) is a device int64 read
 * instead of `step` (CUDA-graph replay: the counter is advanced by the train kernel); lr_dev (nullable) is a device
 * double read instead of `lr`, so a captured graph follows the reference's per-epoch learning-rate decay
 * (adjust_learning_rate, steps/utils.py:301-307, called at steps/traintest.py:83-84) without a re-capture. */
int b2h_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, double lr,
                  double beta1, double beta2, double eps, int64_t step, const int64_t* step_dev, const double* lr_dev,
                  float grad_scale, void* packed, int n_in, int C, int pos_emb, void* stream);

/* ---- data parallel over peer (NVLink / NVSwitch) memory -----------------------------------------------------
 * The reference is single-process; training shards by batch with ONE gradient exchange per step (SURVEY.md §8e) over
 * peer memory, no NCCL call on the step path.  Every rank owns a symmetric exchange buffer (peer-mapped, e.g.
 * torch.distributed._symmetric_memory) whose first index is the epoch parity: a rank one step ahead of a peer never
 * writes words the peer is still reading. */
/* floats a rank's exchange buffer must hold for b2h_train_step_dp */
int64_t b2h_dp_exchange_floats(int n_in, int C, int pos_emb, int world);
/* 32-bit pattern every word of the exchange buffer must be filled with ONCE, before the first step, on every rank:
 * 0xFFFFFFFF for shapes the one-launch tile kernel serves (its exchange words are 4 bytes: the gradient value is its own
 * arrival flag, "not arrived" = this NaN pattern, re-armed by the reader), 0 for the three-launch path (gradients + flags). */
int64_t b2h_dp_exchange_fill(int T, int n_in, int C, int pos_emb, int precision);

/* The whole data-parallel step as ONE call; every rank sums the ranks' gradients in rank order, so the replicas stay
 * bit-identical.  Two paths, by shape (b2h_kernel_choice with train = 1):
 * - B2H_KERNEL_TC_TILE: ONE cooperative launch per rank: forward + loss + backward, grid barrier, cross-CTA reduction,
 *   exchange, Adam + re-pack.  Buffer: 4-byte words [2][world (source rank)][gradient slots], pushed into every rank's
 *   buffer; a word is the fp32 gradient and its own arrival flag (see b2h_dp_exchange_fill).  multicast_buf (nullable):
 *   the multicast (NVLS) address of the buffers (torch symmetric-memory handle .multicast_ptr): ONE multimem.st per slot,
 *   replicated by the NVSwitch, instead of `world` unicast stores.
 * - other shapes: three launches: the train kernel, the reduction into this rank's buffer, and a kernel that stores the
 *   epoch into this rank's flag in every peer's buffer, waits for all flags of its own buffer and sums the peers'
 *   gradients over NVLink before Adam + re-pack.  Buffer: [2][P] fp32 flat gradients, then [world] int64 flags.
 * sym_grads: this rank's buffer; peer_bufs_dev: device array [world] of the ranks' buffers, indexed by rank.
 * step_dev / epoch_dev: device int64 counters advanced by the train kernel (epoch_dev is never rewound).  lr_dev: see
 * b2h_adam_step.  A wait for a peer that exceeds ~3 s sets the status read by b2h_tc_status / b2h_dp_status and
 * suppresses every parameter update until it is read. */
int b2h_train_step_dp(const void* x, int x_dtype, const float* target, const float* conf, const int32_t* lengths,
                      float* params, void* packed, float* exp_avg, float* exp_avg_sq, float* loss_out, int B, int T,
                      int n_in, int C, int pos_emb, int loss_kind, int precision, double lr, double beta1, double beta2,
                      double eps, int64_t* step_dev, int64_t* epoch_dev, const double* lr_dev, float* sym_grads,
                      const void* peer_bufs_dev, void* multicast_buf, int rank, int world, float grad_scale, void* workspace,
                      int64_t workspace_bytes, void* stream);
/* 0 = clean, 1 = a peer-flag wait gave up (bounded spin); reading clears it.  Synchronises the device. */
int b2h_dp_status(void);

/* Fast path = b2h_train_forward_backward + b2h_adam_step with the cross-CTA gradient reduction
 * fused into the Adam kernel (2 launches per step, zero host work); in bf16 mode with step_dev the reduction and
 * Adam run in the tail of the SAME cooperative launch (1 launch per step; the workspace must be zero-initialised
 * once when it is allocated: its first 1024 bytes hold the launch sequence number and the per-CTA arrival flags of
 * the in-kernel grid barrier, at a fixed offset whatever (B, T) is).  step_dev (nullable): a device
 * int64 holding the number of steps taken so far; when given it is incremented on the device and
 * used instead of `step`, so a captured CUDA graph of this call can be replayed step after step. */
int b2h_train_step(const void* x, int x_dtype, const float* target, const float* conf, const int32_t* lengths,
                   float* params, void* packed, float* exp_avg, float* exp_avg_sq, float* loss_out, int B, int T,
                   int n_in, int C, int pos_emb, int loss_kind, int precision, double lr, double beta1,
                   double beta2, double eps, int64_t step, int64_t* step_dev, const double* lr_dev, void* workspace,
                   int64_t workspace_bytes, void* stream);

/* b2h_train_step over window views of frame streams (the streams, crop rule, alignment and served shapes of
 * b2h_train_forward_backward_windows; every other argument as in b2h_train_step).  Bit-identical to b2h_train_step on the
 * materialised windows: loss, params, exp_avg, exp_avg_sq and the packed buffer. */
int b2h_train_step_windows(const void* frames, int x_dtype, const float* target_frames, const float* conf_frames,
                           int64_t n_frames, const int64_t* win_start, const int64_t* win_end, int pad_mode,
                           const int32_t* lengths, float* params, void* packed, float* exp_avg, float* exp_avg_sq,
                           float* loss_out, int n_win, int T, int n_in, int C, int pos_emb, int loss_kind, int precision,
                           double lr, double beta1, double beta2, double eps, int64_t step, int64_t* step_dev,
                           const double* lr_dev, void* workspace, int64_t workspace_bytes, void* stream);

/* tcgen05 / TMEM / descriptor self-test (tests/test_tc_probe.py): D = A·B^T for one 128xNx(16*ksteps)
 * bf16 tile staged in the no-swizzle K-major layout the conv kernels use, A rows shifted by `shift`
 * rows (the implicit-im2col trick).  out (128,N) fp32. */
int b2h_tc_probe(const void* a_bf16, const void* b_bf16, float* out, int n, int ksteps, int shift, int variant,
                 void* stream);

/* device-side wait-timeout status of the tensor-core kernels: 0 = clean, else the id of the wait that
 * gave up (the kernels never spin forever); reading clears it.  Synchronises the device. */
int b2h_tc_status(void);

/* Bring-up aid (microbenchmarks behind DESIGN.md's pacing numbers; tools/tc_bench*.py, tools/tma_bench.py).
 * M = 64 | 128: cycles for `reps` back-to-back tcgen05.mma (bf16, K=16) of shape MxN rotating over `nacc & 255`
 *   accumulators, issued from `nacc >> 8` warps (0 = 1); out[0] = issue-to-completion cycles, out[1] = issue-loop cycles.
 *   `mn_major` bit 0: MN-major operands; bit 1: 128B-swizzle descriptors (timing only); bit 2: walk A rows / B blocks;
 *   bit 3: tcgen05.commit after every second MMA; bit 4: non-zero operand data; bits 5-7: chunk-stride variants;
 *   bits 8..: number of CTAs (0 = 1).
 * M = 1: steady-state L2 -> shared throughput of 1-D cp.async.bulk copies: N = bytes per copy (divides 8192),
 *   reps = rounds, nacc = ring depth in 8-KB stages (<= 16), mn_major = CTAs; out[0] = cycles, out[1] = bytes. */
int b2h_tc_bench(void* out_i64x2, int M, int N, int reps, int nacc, int mn_major, void* stream);

/* Bring-up aid: when set to a device buffer of 1024 int64, CTA 0 of the tile kernels stamps clock64() at every
 * phase boundary (setup, staging, per-layer issue / ready / epilogue) into words [0, 128), and every CTA c of the fused
 * train kernel writes %globaltimer (ns) at its start / barrier arrival / barrier exit / end into words
 * [128 + 4c, 128 + 4c + 4); NULL switches it off. */
void b2h_debug_timing(void* dev_i64x1024);

/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t b2h_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B2H_H_ */
