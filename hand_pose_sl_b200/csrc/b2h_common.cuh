// Shared geometry / helpers for libb2h.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "../../include/b2h.h"

#define B2H_KW 5          // kernel_size of every Conv1d (HandPoseModels.py:24-32)
#define B2H_PADW 2        // padding=2
#define B2H_COUT 42       // 2*21 output channels (HandPoseModels.py:32)
#define B2H_MAX_C 256

namespace b2h {

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Layout of the flat fp32 parameter buffer (state_dict order) and of the packed weight buffer.
struct Geo {
  int n_in, C, pos_emb;     // pos_emb: 0 / 1 (the positional row t / pe_len in front of the input channels)
  int pe_len;               // LinearPositionalEmbedding(max_len): 100 in the reference (HandPoseModels.py:23)
  int cin[4], cout[4];
  int w_off[4], b_off[4];   // float offsets into the flat parameter buffer
  int P;                    // total parameter count
  // packed buffer (byte offsets, each 128-B aligned)
  int64_t wf_off[4];        // fp32 forward taps   Wf[k][ci][co]            = W[co][ci][k]
  int64_t wd_off[4];        // fp32 dgrad taps     Wd[k'][co][ci]           = W[co][ci][4-k']   (layers 2..4)
  int64_t tf_off[4];        // bf16 UMMA B operand, forward  (blocks of [2][N][8])
  int64_t td_off[4];        // bf16 UMMA B operand, dgrad    (layers 2..4)
  int64_t tfl_off[4];       // bf16 UMMA B operand, forward, LOW halves: w - bf16(w) rounded to bf16 (fp32 mode on tcgen05:
                            // x*w ~ x_hi*w_hi + x_lo*w_hi + x_hi*w_lo with fp32 accumulation, ~6e-6 relative)
  int64_t bias_off;         // fp32 [4][64] zero-padded biases (one 1-KB bulk copy into smem)
  int kp[4], np_[4];        // UMMA padded reduction (cin -> mult of 16) and N (cout -> mult of 16), forward
  int64_t packed_bytes;
};

__host__ __device__ inline Geo make_geo(int n_in, int C, int pos_emb) {
  Geo g;
  // `pos_emb` of the C-ABI: 0 = off, 1 = on with the reference's max_len = 100, n > 1 = on with max_len = n
  g.n_in = n_in; g.C = C; g.pos_emb = pos_emb ? 1 : 0; g.pe_len = pos_emb > 1 ? pos_emb : 100;
  g.cin[0] = n_in + (pos_emb ? 1 : 0); g.cout[0] = C;
  g.cin[1] = C; g.cout[1] = C;
  g.cin[2] = C; g.cout[2] = C;
  g.cin[3] = C; g.cout[3] = B2H_COUT;
  int off = 0;
  for (int l = 0; l < 4; ++l) {
    g.w_off[l] = off; off += g.cout[l] * g.cin[l] * B2H_KW;
    g.b_off[l] = off; off += g.cout[l];
  }
  g.P = off;
  int64_t b = 0;
  for (int l = 0; l < 4; ++l) { g.wf_off[l] = b; b += (int64_t)B2H_KW * g.cin[l] * g.cout[l] * 4; b = (b + 127) / 128 * 128; }
  for (int l = 0; l < 4; ++l) { g.wd_off[l] = b; if (l > 0) { b += (int64_t)B2H_KW * g.cin[l] * g.cout[l] * 4; b = (b + 127) / 128 * 128; } }
  for (int l = 0; l < 4; ++l) {
    g.kp[l] = round_up(g.cin[l], 16); g.np_[l] = round_up(g.cout[l], 16);
    g.tf_off[l] = b; b += (int64_t)B2H_KW * g.kp[l] * g.np_[l] * 2; b = (b + 127) / 128 * 128;
  }
  for (int l = 0; l < 4; ++l) {
    g.td_off[l] = b;
    if (l > 0) { b += (int64_t)B2H_KW * round_up(g.cout[l], 16) * round_up(g.cin[l], 16) * 2; b = (b + 127) / 128 * 128; }
  }
  for (int l = 0; l < 4; ++l) { g.tfl_off[l] = b; b += (int64_t)B2H_KW * g.kp[l] * g.np_[l] * 2; b = (b + 127) / 128 * 128; }
  g.bias_off = b; b += 4 * 64 * 4;
  g.packed_bytes = b;
  return g;
}

// Byte offset inside one UMMA B-operand section of element (n, kk) of tap k.
// Section = blocks q = k*(KP/16)+s of [2 k-chunks][N rows][8 bf16] (no-swizzle K-major canonical
// layout: core matrix = 8 rows x 16 B, SBO = 128 B between 8-row groups, LBO = N*16 B between chunks).
__host__ __device__ inline int64_t umma_b_offset(int k, int kk, int n, int KP, int N) {
  int s = kk >> 4, chunk = (kk >> 3) & 1, within = kk & 7;
  int64_t q = (int64_t)k * (KP >> 4) + s;
  return q * ((int64_t)N * 32) + (int64_t)chunk * (N * 16) + (int64_t)n * 16 + within * 2;
}

// Gradient-partial layout written by every training kernel (tile, wide wgrad, FFMA).  The TMEM read-out has lane =
// output channel and 32 consecutive columns = input channels, so the W part is stored [k][ci/4][co][4 ci]: for a fixed
// (k, ci/4) the lanes of a warp store consecutive float4s (coalesced; the [k][co][ci] order of round 1 made every lane
// of a store instruction hit its own 128-B line: ~6k cycles of read-out per CTA).  The FFMA kernel's lanes are output
// channels too: for a fixed (k, ci) its stores are 16 B apart.
//   per layer l: W part [k][kp_l/4][cout_l][4] then bias part [cout_l] (padded to a multiple of 4)
// The slots with ci >= cin and the bias padding carry no parameter: writers may leave them unwritten, readers decode
// them as padding (gp_decode / flat_index_of_gp) and never apply them.
__host__ __device__ inline int gp_layer_size(const Geo& g, int l) { return B2H_KW * g.cout[l] * g.kp[l] + round_up(g.cout[l], 4); }
__host__ __device__ inline int gp_layer_off(const Geo& g, int l) {
  int o = 0;
  for (int q = 0; q < l; ++q) o += gp_layer_size(g, q);
  return o;
}
__host__ __device__ inline int gp_total(const Geo& g) { return gp_layer_off(g, 4); }

// (layer, tap, co, ci) of one parameter; is_bias: co = bias index, k = ci = 0
struct GpSlot { int l, k, co, ci; bool is_bias; };
// slot of weight (s.l, s.k, s.ci, s.co) or of bias (s.l, s.co) inside layer s.l's part of a slice (add gp_layer_off)
__host__ __device__ inline int gp_slot_in_layer(const Geo& g, const GpSlot& s) {
  const int l = s.l;
  if (s.is_bias) return B2H_KW * g.cout[l] * g.kp[l] + s.co;
  return ((s.k * (g.kp[l] >> 2) + (s.ci >> 2)) * g.cout[l] + s.co) * 4 + (s.ci & 3);
}
// flat parameter index -> slot
__host__ __device__ inline GpSlot gp_slot_of_flat(const Geo& g, int i) {
  GpSlot s;
  int l = 0;
  for (int q = 1; q < 4; ++q)
    if (i >= g.w_off[q]) l = q;
  s.l = l;
  if (i >= g.b_off[l]) { s.is_bias = true; s.k = 0; s.ci = 0; s.co = i - g.b_off[l]; return s; }
  s.is_bias = false;
  const int cin = g.cin[l];
  const int rel = i - g.w_off[l];
  s.co = rel / (cin * B2H_KW);
  const int rem = rel - s.co * cin * B2H_KW;
  s.ci = rem / B2H_KW; s.k = rem - s.ci * B2H_KW;
  return s;
}
// flat parameter index -> index in the GP layout
__host__ __device__ inline int gp_index_of_flat(const Geo& g, int i) {
  const GpSlot s = gp_slot_of_flat(g, i);
  return gp_layer_off(g, s.l) + gp_slot_in_layer(g, s);
}

// GP index -> slot.  Returns false for the padding slots.
__host__ __device__ inline bool gp_decode(const Geo& g, int j, GpSlot& s) {
  int l = 0, base = 0;
  for (int q = 0; q < 4; ++q) {
    const int sz = gp_layer_size(g, q);
    if (j >= base + sz && q < 3) { base += sz; l = q + 1; }
    else break;
  }
  const int rel = j - base;
  const int wsz = B2H_KW * g.cout[l] * g.kp[l];
  s.l = l;
  if (rel >= wsz) { s.is_bias = true; s.k = 0; s.ci = 0; s.co = rel - wsz; return s.co < g.cout[l]; }
  s.is_bias = false;
  const int e = rel & 3;
  int r = rel >> 2;
  const int q4 = g.kp[l] >> 2;
  s.co = r % g.cout[l]; r /= g.cout[l];
  const int qq = r % q4;
  s.k = r / q4;
  s.ci = 4 * qq + e;
  return s.ci < g.cin[l];
}
__host__ __device__ inline int gp_flat_of_slot(const Geo& g, const GpSlot& s) {
  return s.is_bias ? g.b_off[s.l] + s.co : g.w_off[s.l] + (s.co * g.cin[s.l] + s.ci) * B2H_KW + s.k;
}
// GP index -> flat parameter index (-1 for the padding slots of the GP layout)
__host__ __device__ inline int flat_index_of_gp(const Geo& g, int j) {
  GpSlot s;
  return gp_decode(g, j, s) ? gp_flat_of_slot(g, s) : -1;
}

// Scatter one fp32 parameter into the packed operand layouts (callers holding a flat index decode it with gp_slot_of_flat).
__device__ __forceinline__ void scatter_packed(const Geo& g, char* packed, const GpSlot& s, float v) {
  const int l = s.l;
  if (s.is_bias) {              // bias: also kept zero-padded [4][64] for the tensor-core kernels' smem copy
    if (s.co < 64) reinterpret_cast<float*>(packed + g.bias_off)[l * 64 + s.co] = v;
    return;
  }
  const int cin = g.cin[l], cout = g.cout[l], co = s.co, ci = s.ci, k = s.k;
  reinterpret_cast<float*>(packed + g.wf_off[l])[(k * cin + ci) * cout + co] = v;
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  const int64_t bo = umma_b_offset(k, ci, co, g.kp[l], g.np_[l]);
  *reinterpret_cast<__nv_bfloat16*>(packed + g.tf_off[l] + bo) = h;
  *reinterpret_cast<__nv_bfloat16*>(packed + g.tfl_off[l] + bo) = __float2bfloat16_rn(v - __bfloat162float(h));
  if (l > 0) {
    reinterpret_cast<float*>(packed + g.wd_off[l])[((B2H_KW - 1 - k) * cout + co) * cin + ci] = v;
    *reinterpret_cast<__nv_bfloat16*>(packed + g.td_off[l] +
                                      umma_b_offset(B2H_KW - 1 - k, co, ci, round_up(cout, 16), round_up(cin, 16))) = h;
  }
}

// torch.optim.Adam single-tensor update of one element (defaults: amsgrad=False, weight_decay=0, maximize=False) with the
// already scaled gradient gr:
//   m.lerp_(g, 1-b1); v.mul_(b2).addcmul_(g, g, 1-b2);
//   denom = v.sqrt()/sqrt(1-b2^t) + eps;  p.addcdiv_(m, denom, value=-lr/(1-b1^t))
// m and v are updated in place; returns the new p.  step_size = lr/(1-b1^t), inv_bc2_sqrt = 1/sqrt(1-b2^t).
__device__ __forceinline__ float adam_update(float& m, float& v, float p, float gr, float one_minus_b1, float one_minus_b2,
                                             float beta2, float eps, float step_size, float inv_bc2_sqrt) {
  m = fmaf(gr - m, one_minus_b1, m);
  v = fmaf(one_minus_b2 * gr, gr, v * beta2);
  const float denom = sqrtf(v) * inv_bc2_sqrt + eps;
  return p - step_size * (m / denom);
}

// beta^t for an integer step count by binary exponentiation (~2*log2(t) DMULs instead of a double-precision pow())
__host__ __device__ inline double ipow(double b, long long t) {
  double r = 1.0;
  while (t > 0) {
    if (t & 1) r *= b;
    b *= b;
    t >>= 1;
  }
  return r;
}

// Sub-window decomposition of a training window (see TcTileArgs in b2h_train_tc.cuh): window frames [0, T) are cut into
// n_sub cores [cb_i, cb_{i+1}): the first core takes Ts - 16 frames, every further one Ts - 32 (the last: what is left);
// sub-window i covers Ts frames from `start` = cb_i - 16 clamped to [0, T - Ts], so that every interior cut has >= 16 real
// frames of context on both sides.  Core rows in sub-window coordinates: [clo, chi).
struct SubWindow { int start, clo, chi; };
__host__ __device__ inline int sub_window_cut(int T, int Ts, int n_sub, int i) {
  if (i <= 0) return 0;
  if (i >= n_sub) return T;
  const int c = (Ts - 16) + (i - 1) * (Ts - 32);
  return c < T ? c : T;
}
__host__ __device__ inline SubWindow sub_window(int T, int Ts, int n_sub, int i) {
  SubWindow s;
  const int cb0 = sub_window_cut(T, Ts, n_sub, i), cb1 = sub_window_cut(T, Ts, n_sub, i + 1);
  int st = cb0 - 16;
  st = st < 0 ? 0 : st;
  st = st > T - Ts ? T - Ts : st;
  s.start = st; s.clo = cb0 - st; s.chi = cb1 - st;
  return s;
}
// Number of sub-windows of Ts frames the cut rule above makes of a sequence of L frames (n_sub of sub_window): 0 for an empty
// one, 1 for L <= Ts (one sub-window, core [0, L)), otherwise the least n >= 2 whose cores (Ts - 16) * 2 + (n - 2) * (Ts - 32)
// = n (Ts - 32) + 32 frames cover L.  So n <= 1 + L / (Ts - 32) for every L, and a set of sequences with F frames in all
// is cut into at most n_seq + F / (Ts - 32) sub-windows (the bound that sizes the utterance forward's grid and workspace).
__host__ __device__ inline int sub_window_count(long long L, int Ts) {
  if (L <= 0) return 0;
  if (L <= Ts) return 1;
  const long long n = (L - 32 + (Ts - 32) - 1) / (Ts - 32);
  return n < 2 ? 2 : (int)n;
}

// Workspace header of the fused train kernel (first B2H_WS_HEADER bytes of the caller's workspace, zeroed once when the
// workspace is allocated and owned by the kernels afterwards; FIXED offset, so runners of different (B, T) that share
// one workspace can never find gradient partials where they expect barrier words):
//   u32 [0]        launch sequence number (read by every CTA at kernel start, advanced by CTA 0 after the grid barrier)
//   u32 [4 + c]    arrival flag of CTA c (= sequence number of the launch it last arrived in)
#define B2H_WS_HEADER 1024
#define B2H_WS_MAX_CTA 192

// Optional tail of the tensor-core train kernel: cross-CTA gradient reduction, (data-parallel) gradient exchange
// over peer memory and Adam, all inside the SAME cooperative launch (grid barrier through the workspace header).
struct FuseAdam {
  int enabled;
  float* params; float* m; float* v; char* packed;
  double lr, beta1, beta2;
  const double* lr_dev;              // nullable: learning rate read from device memory (a captured graph follows lr changes)
  float eps, grad_scale;
  const long long* step_dev;
  float* loss_out;
  unsigned* hdr;                     // workspace header (B2H_WS_HEADER bytes)
  // data parallel (world > 1)
  const float* const* peer_bufs;     // device array [world] of peer exchange buffers
  float* sym_grads;                  // this rank's exchange buffer
  unsigned long long* mc_buf;        // nullable: multicast (NVLS) address of the exchange buffers: one multimem.st reaches every rank
  const long long* epoch_dev;
  int rank, world;
};

void set_error(const char* fmt, ...);
int check_launch(const char* what);
void count_launch(int n = 1);


// Streaming inference (BASELINE config 5) and training from device-resident streams: sliding windows read as views of a
// per-frame stream (n_frames, n_in) -- and, in training, of the target (n_frames, 42) and confidence (n_frames, 21) streams
// at the same rows -- instead of materialised (n_win, T, .) windows.  win_start == nullptr: the kernel's inputs are dense.
struct WindowView { const long long* win_start; const long long* win_end; long long n_frames; int pad_mode; };

// Source row in the stream of (window w, frame t) of a window view; -1 = a zero row.  The crop [start, start + T) is cut at
// min(win_end[w], n_frames) (win_end nullable), then the dataset's pad rule fills the rest (repeat the crop's first frame:
// text_pose_dataset.py:511-518; zeros: :614-622) -- the same integer work as K0's windowing (b2h_preprocess.cu), so a view
// reads exactly the rows K0 would materialise.  The tile kernel keeps the same rule inline (xrow_of, b2h_train_tc.cuh):
// calling this function there changes the register allocation of its NT = 1 instantiations.
__device__ __forceinline__ long long window_src_row(const WindowView& v, int w, int t) {
  const long long start = v.win_start[w];
  long long cend = v.win_end ? v.win_end[w] : v.n_frames;
  cend = cend > v.n_frames ? v.n_frames : cend;
  long long f = start + t;
  if (f >= cend || f < 0) f = (v.pad_mode == B2H_PAD_REPEAT_FIRST && start >= 0 && start < cend) ? start : -1;
  return f;
}

// Utterances and segments (host side; the planning kernel turns them into the table of UttPlan): sequence s of n is stream
// rows [seg_a[s], seg_b[s]), predicted or trained as one sequence.  The forward's offsets are (off, off + 1, n_utt, n_frames,
// max_len = 0); training and validation segments hold 1..max_len frames each.
struct SegmentView { const long long* seg_a; const long long* seg_b; int n; long long n_frames; int max_len; };

// ---- launch plans: for each kernel family, one host function (in the file that owns the kernel) decides whether a
// shape fits and how it launches.  The C-ABI queries, the workspace layout and the launchers all read the same plan, so
// the number of gradient / loss partial slices a launch writes is the number the workspace was sized for. ----

// Tile kernel (b2h_train_tc.cuh): weights resident in shared memory, independent 64/128/256-row tiles.
struct TilePlan {
  bool ok, train, split;    // split = fp32 mode on the tensor pipe (bf16 high/low operand pairs)
  int n_sub;                // training sub-windows per window (1 = whole windows; see TcTileArgs)
  int B, T;                 // launch batch and window length: B * n_sub sub-windows of T = 128 (split) / 256 frames if n_sub > 1
  int nhalf, MB, NT, HR, gh, n_tiles;
  size_t smem;
  int grid;                 // CTAs = gradient and loss partial slices of a training launch
};
TilePlan plan_tile(const Geo& g, int B, int T, bool train, bool split);

// Row-space forward (b2h_conv_tc.cu): G windows per CTA in one layer-major row space of NT 128-row tiles.
struct RowspacePlan {
  bool ok;                  // one window per CTA fits: support does not depend on B
  int G, NT, RBUF;
  size_t smem;
  int grid;
};
RowspacePlan plan_rowspace(const Geo& g, int B, int T);

// Wide kernels (b2h_wide_tc.cuh): weights streamed through a ring of nstage stages; training adds split-K wgrad.
struct WidePlan {
  bool ok;
  int gh, n_tiles, a_bytes, nstage;
  size_t smem;
  int grid;
  int ksplit;               // training: gradient partial slices written by the wgrad kernel
  int n_loss;               // training: loss partials (one per CTA of the forward+criterion kernel)
  int64_t scratch_bytes;    // training: per-tile operand dumps
};
WidePlan plan_wide(const Geo& g, int B, int T);

// FFMA kernel (b2h_conv_fp32.cu): one window per CTA iteration, fp32 activations in shared memory.
struct FfmaPlan {
  bool ok, train;
  size_t smem;
  int grid;                 // training: CTAs = gradient and loss partial slices
};
FfmaPlan plan_ffma(const Geo& g, int B, int T, bool train);

// ---- the request block of every forward / training launch, and the launchers ----
// Filled once by the C-ABI entry points; each launcher copies what its kernel needs into that kernel's own parameter
// block.  Its layout is also conv_fp32_kernel's parameter block.
struct ConvArgs {
  const void* x; int x_dtype;
  const float* target; const float* conf; const float* d_y; const int32_t* lengths;
  const float* params; const char* packed;
  float* y;                 // forward output / masked prediction (nullable in train mode)
  float* partials;          // [grid][gp_total]
  float* loss_partials;     // [grid]; a forward over utterances: nullptr, or one criterion sum per sub-window (validation)
  long long* step_dev;      // nullable: device step counter, incremented by block 0 (read by the Adam kernel)
  long long* epoch_dev;     // nullable: data-parallel exchange epoch, incremented the same way (never rewound)
  FuseAdam fuse;            // tensor-core train kernel only: reduce + exchange + Adam in the same launch
  int B, T, loss_kind, apply_mask, mode;   // mode 0 = forward, 1 = train (loss inside), 2 = backward of given d_y
  float out_scale;
  Geo geo;
  WindowView wv;            // tensor-core kernels only: win_start set = x (and target / conf) are frame streams, B = windows
  const int4* utt;          // forward over utterances (b2h_utterances.cuh): the device-side plan, x a frame stream; else nullptr
  const int2* utt_seg;      // training over segments: per sub-window {segment, segment length} (UttPlan); else nullptr
  int utt_max_len;          // training over segments: row stride of the masked prediction (n_seg, max_len, 42)
};
int launch_fp32(const ConvArgs& a, const FfmaPlan& plan, cudaStream_t stream);
int launch_tc_fwd(const ConvArgs& a, const RowspacePlan& plan, cudaStream_t stream);
// forward (mode 0) or training; the tile kernel takes its launch batch and window length from the plan
int launch_tc_tile(const ConvArgs& a, const TilePlan& plan, cudaStream_t stream);
int launch_tc_wide_fwd(const ConvArgs& a, const WidePlan& plan, cudaStream_t stream);
// wide training (32 < conv_channels <= 256, bf16 mode): forward+criterion / dgrad chain / split-K wgrad over the per-tile
// operand dumps in `scratch` (workspace past the partials, TrainPlan::scratch_off)
int launch_tc_wide_train(const ConvArgs& a, const WidePlan& plan, unsigned char* scratch, cudaStream_t stream);
int launch_tc_probe(const void* a, const void* b, float* out, int n, int ksteps, int shift, int variant, cudaStream_t stream);
int tc_status_and_clear();

// Forward over packed utterances (b2h_conv_forward_utterances): every utterance is cut into sub-windows of Ts frames by
// sub_window(); the forward kernels read sub-window g from a table that a one-CTA planning kernel builds on the device.
// One workspace layout for the forward, training and validation, from the table at plan_off (0 unless training, where the
// header and the gradient and loss partials of the plan's grid come first):
//   [int4 {sub-window count, bad, 0, 0}][int4 per sub-window, max_sub of them][int prefix[n + 1]]
//   segments (training, validation): at seg_off, the next 16-byte boundary, one int2 {segment, segment length} per sub-window
//   validation: at part_off, right after them, one float per sub-window: its criterion sum, written by the forward
// and the whole rounded up to 256 B.  Sub-window g = {stream row of its first frame, its first frame in the sequence,
// clo | chi << 16, frames before the sequence end (<= Ts)}; bad = 1 when the planning kernel refused the offsets / segments
// (count = 0 then).
struct UttPlan {
  int kernel;               // B2H_KERNEL_TC_TILE | B2H_KERNEL_TC_WIDE | B2H_KERNEL_NONE
  int Ts;                   // sub-window length
  int max_sub;              // upper bound on the sub-window count: n_utt + n_frames / (Ts - 32); segments: n_seg * n(max_len)
  TilePlan tile; WidePlan wide;   // planned for max_sub windows of Ts frames
  int64_t ws_bytes;
  int64_t plan_off;         // byte offset of the table in the workspace
  int64_t seg_off, part_off;  // byte offsets of the segment pairs and of the per-sub-window sums from the table
};
__host__ __device__ inline int64_t utt_prefix_offset(int max_sub) { return (int64_t)(1 + max_sub) * 16; }
// The planning kernel over the sequences of `sv` into `table` (the workspace at plan.plan_off), then the kernel the plan
// names over the table it wrote: training (a.mode 1) the tile kernel with a.B = sv.n segments (a.fuse.enabled: the fused
// step); the forward the tile or wide kernel with a.B = plan.max_sub sub-windows; validation (the forward with
// a.loss_partials = the per-sub-window sums) that forward, then the kernel that writes seg_loss (nullable) and *loss_out.
int launch_utterances(ConvArgs a, const UttPlan& plan, const SegmentView& sv, void* table, float* seg_loss, float* loss_out,
                      cudaStream_t stream);

void set_debug_timing(long long* p);
int launch_format_prediction(const float* pred, float* out, int64_t rows, int mode, cudaStream_t stream);
int launch_pos_emb_concat(const float* inp, float* out, int B, int Cc, int T, int max_len, cudaStream_t stream);
int launch_pack(const float* params, void* packed, const Geo& g, cudaStream_t stream);
// grads (flat parameter order) = sum of the nparts gradient-partial slices; *loss_out = sum of the n_loss loss partials
int launch_reduce(const float* partials, int nparts, const Geo& g, float* grads, const float* loss_partials, int n_loss,
                  float* loss_out, const long long* epoch_dev, cudaStream_t stream);
int launch_adam_dp(float* params, const float* const* peer_bufs, int rank, int world, float* m, float* v, int64_t n, double lr,
                   double beta1, double beta2, double eps, const long long* step_dev, const long long* epoch_dev, const double* lr_dev,
                   float grad_scale, void* packed, const Geo& g, cudaStream_t stream);
int dp_status_and_clear();
// Adam on the sum of the nparts gradient-partial slices a training launch left in the workspace (+ the loss sum)
int launch_adam_partials(float* params, const float* partials, int nparts, float* m, float* v, double lr, double beta1,
                         double beta2, double eps, int64_t step, const long long* step_dev, const double* lr_dev, void* packed,
                         const Geo& g, const float* loss_partials, int n_loss, float* loss_out, cudaStream_t stream);
// Adam on an already-reduced gradient of n parameters in flat order (b2h_adam_step); packed == nullptr: no re-pack
int launch_adam_flat(float* params, const float* grads, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                     double eps, int64_t step, const long long* step_dev, const double* lr_dev, float grad_scale, void* packed,
                     const Geo& g, cudaStream_t stream);
int launch_mask_output(float* y, const int32_t* lengths, int B, int T, int row, cudaStream_t stream);
int launch_pose_l1(const float* pred, const float* target, const float* scores, const int32_t* lengths, int B, int T, int row,
                   int loss_kind, float* loss_out, float* d_pred, float* row_scratch, cudaStream_t stream);
int num_sms();                                        // SM count of the CURRENT device (cached per device)
// cudaFuncAttributeMaxDynamicSharedMemorySize for `fn` on the CURRENT device, raised on demand; the cache is keyed by
// (function, device) so that one process can drive several GPUs (inference replicas).  Returns B2H_OK / B2H_ECUDA.
int ensure_dyn_smem(const void* fn, size_t bytes);

}  // namespace b2h
