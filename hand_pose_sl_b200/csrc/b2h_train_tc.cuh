// bf16 mode, tile kernel: forward (+ masked-L1 loss + full backward) of independent 128-row tiles on
// tcgen05 / TMEM.  Included by b2h_conv_tc.cu (same translation unit as the PTX layer).
//
// Reference semantics (paths relative to the reference root):
//   ConvModel.forward                 body2hand/src/models/HandPoseModels.py:40-64
//   mask_output                       body2hand/src/steps/utils.py:309-312
//   maskedPoseL1 / poderatedPoseL1    body2hand/src/steps/utils.py:413-452
//   loss.backward()                   body2hand/src/steps/traintest.py:120
//
// Tile geometry.  A tile is 128 TMEM lanes of output rows made of `nhalf` independent row segments:
//   mode B (T <= 64): two segments of 64 rows, one M=64 MMA each (TMEM lanes 32q+i and 32q+16+i), every
//                     segment holding g = floor(66/(T+2)) whole windows -> T=64: 2 windows per tile, no
//                     padded-row waste; the two segments are issued by two different warps;
//   mode A (64 < T <= 256): one segment of 128*NT rows (NT = 1 for T <= 128, else 2), one window, NT M=128 MMAs per
//                     conv tap issued by NT warps into NT accumulators (TMEM columns 64j); every thread then owns NT rows.
// A segment lives in shared memory as [2 zero rows][window][2 zero rows][window]...[zero rows] in the
// no-swizzle K-major canonical layout [channel/8][row][8 ch] (16-B rows), so conv tap k is a +k change of
// the A descriptor's start-address field and the SAME buffer also serves, read as an MN-major operand, as
// A (dZ^T) or B (layer input) of the weight-gradient GEMM (reduction over frames).
//
// Per tile: F1 F2 F3 F4(+loss,+dY) | D4,W4 | D3,W3 | D2,W2 | W1.   F/D = conv GEMM + epilogue
// (tcgen05.ld -> bias/ReLU or ReLU-mask -> bf16 -> st.shared); W = weight/bias-gradient GEMMs that keep
// accumulating in TMEM across all tiles of the CTA and are read out once at the end into the CTA's slice of the
// partials workspace (deterministic 2-stage sum).  In the backward warps 0/1 only issue MMAs and warps 2..7 run the
// D epilogues, each under the W GEMMs issued right after its D, so the tensor pipe runs D4 W4 D3 W3 D2 W2 W1 back to
// back; an mbarrier handshake (not __syncthreads) tells the issuers that the next D's operand is ready.
//
// Measured on B200: one tcgen05.mma costs >= ~25 (M=64) / ~40 (M=128) cycles whatever N <= 64 is, so the MMA
// phases are instruction-count bound at C=30: descriptors are pre-encoded (one integer add per MMA) and the
// two row segments are issued from two warps.
// Data movement: weights + biases by 1-D TMA bulk copies (cp.async.bulk, once per CTA), the target tile by bulk
// copies (prefetched at tile start), the prediction tile by bulk stores; inputs are prefetched into registers
// one tile ahead (fp32 -> bf16 conversion happens on the way to shared memory).
#pragma once
#include <type_traits>

namespace b2h {
using namespace tc;

struct TcTileArgs {
  const void* x; int x_dtype;
  const float* target; const float* conf; const float* d_y; const int32_t* lengths;
  const float* params; const char* packed;
  float* y;               // forward output / masked prediction (nullable in train mode)
  float* partials;        // [grid][GP]  (gradient-partial layout, b2h_common.cuh gp_*)
  float* loss_partials;   // [grid]
  long long* step_dev;
  long long* epoch_dev;
  long long* dbg;         // nullable: CTA 0 / thread 0 writes clock64() phase stamps here (b2h_debug_timing)
  FuseAdam fuse;
  // Window views (streaming inference; training from device-resident streams): when win_start is set, x is a per-frame
  // stream (n_frames, n_in) and window w, frame t reads row win_start[w] + t of it (cut at win_end[w] / n_frames, then the
  // dataset's pad rule) -- overlapping windows are views of the stream, nothing is re-materialised.  Training reads the
  // target (n_frames, 42) and confidence (n_frames, 21) rows at the same stream row; the prediction stays dense.
  const long long* win_start; const long long* win_end; long long n_frames; int pad_mode;
  // Sub-window training (n_sub > 1: T_orig > 128 in fp32 mode, > 256 in bf16 mode): a tile segment holds 128 (doubled
  // operand buffers) / 256 frames, so every window is processed as n_sub overlapping sub-windows that read REAL neighbouring frames
  // (>= 16 on each interior side) instead of zero padding; the criterion (and d_y) is applied to the sub-window's core
  // rows only.  The backward is linear in d(loss)/d(pred) and the activations are exact up to 8 frames from a cut, so the
  // sum of the sub-windows' weight gradients is the window's gradient.  B / T are then the sub-window count / length.
  int T_orig, n_sub, loss_B;
  int B, T, loss_kind, apply_mask, mode;   // mode 0 = forward only, 1 = train (loss inside), 2 = backward of given d_y
  float out_scale;
  int n_tiles, nhalf, MB, HR, gh, NT;      // tile geometry (NT = 128-row MMA tiles per segment: 2 for 128 < T <= 256)
  Geo geo;
  // Forward over utterances (UTT instantiations): x is a frame stream and window g < utt[0].x is sub-window utt[1 + g] of the
  // plan (UttPlan, b2h_common.cuh); B / n_tiles are the host's upper bound on the sub-window count.
  const int4* utt;
  // Training over segments (TRAIN && UTT): sub-window g belongs to segment utt_seg[g].x of utt_seg[g].y frames (loss weight
  // 1 / (42 L_s), masked-prediction row utt_seg[g].x * utt_max_len + frame); B is the bound on the sub-window count and
  // loss_B the segment count.
  const int2* utt_seg; int utt_max_len;
};

constexpr int kTileThreads = 256;   // 8 warps: two per TMEM lane quadrant (each takes every other 16-column chunk)
constexpr int kAccCol = 0;        // forward / dgrad accumulator: columns [0, 64)
// weight-gradient accumulators follow the forward/dgrad accumulators: 2 layer pairs x (5 taps x 32 + 8 bias) columns
constexpr int kWgPairCols = 5 * 32 + 8;
constexpr int kGatherDepth = 24; // independent 16-B loads in flight per thread in the cross-CTA gradient gather
constexpr uint32_t kDpSentinel = 0xFFFFFFFFu;   // "not arrived yet" in the data-parallel exchange buffer (see the train kernel tail)

struct TileSmem {   // byte offsets into dynamic smem
  int g0, g1, x, a1, a2, a3, ones, lo_off, ys, has_ys, wf[4], wlo_off, wd[4], total;
};

// split = fp32 mode on the tensor pipe: every activation / gradient buffer and every forward weight block exists twice
// (bf16 high half, bf16 low half = bf16(v - high)); the low copies sit at a constant distance (lo_off / wlo_off) behind
// the high ones.  The dgrad operand blocks are not staged in split mode (the forward blocks are read MN-major instead),
// nor is the fp32 staging tile of the training kernel (the target rows are read from global memory).
__host__ __device__ inline TileSmem tile_smem_layout(const Geo& g, int rows, bool train, bool split = false) {
  TileSmem s;
  const int CH = rows * 16;
  int o = 0;
  // gradient buffers first: the M=64 MN-major A operand of the weight-gradient GEMM spans 8 chunks from
  // their start and must stay inside the allocation (the extra chunks only feed ignored accumulator rows)
  s.g0 = o; o += train ? 6 * CH : 0;
  s.g1 = o; o += train ? 4 * CH : 0;
  s.x = o;  o += (g.kp[0] / 8) * CH;
  s.a1 = o; o += (g.kp[1] / 8) * CH;
  s.a2 = o; o += (g.kp[1] / 8) * CH;
  s.a3 = o; o += train ? (g.kp[1] / 8) * CH : 0;
  s.ones = o; o += train ? CH : 0;
  s.lo_off = split ? o : 0;
  if (split) o *= 2;
  s.has_ys = (split && train) ? 0 : 1;
  s.ys = o; o += s.has_ys ? 128 * B2H_COUT * 4 : 0;   // fp32 staging rows: y tile on its way out (fwd) / target tile on its way in (train)
  const int w0 = o;
  for (int l = 0; l < 4; ++l) { s.wf[l] = o; o += B2H_KW * g.kp[l] * g.np_[l] * 2; }
  s.wlo_off = split ? o - w0 : 0;
  if (split) o += o - w0;
  for (int l = 0; l < 4; ++l) {
    s.wd[l] = o;
    if (train && l > 0 && !split) o += B2H_KW * round_up(g.cout[l], 16) * round_up(g.cin[l], 16) * 2;
  }
  s.total = o;
  return s;
}

__device__ __forceinline__ void store8_bf16(unsigned char* buf, int CH, int row, int chunk, const float* v) {
  uint4 q;
  q.x = pack_bf16x2(v[0], v[1]); q.y = pack_bf16x2(v[2], v[3]);
  q.z = pack_bf16x2(v[4], v[5]); q.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(buf + (size_t)chunk * CH + (size_t)row * 16) = q;
}
// split form: high halves to `buf`, low halves bf16(v - high) to buf + lo_off (same position)
template <bool SPLIT>
__device__ __forceinline__ void store8_act(unsigned char* buf, int lo_off, int CH, int row, int chunk, const float* v) {
  uint4 q;
  q.x = pack_bf16x2(v[0], v[1]); q.y = pack_bf16x2(v[2], v[3]);
  q.z = pack_bf16x2(v[4], v[5]); q.w = pack_bf16x2(v[6], v[7]);
  unsigned char* dst = buf + (size_t)chunk * CH + (size_t)row * 16;
  *reinterpret_cast<uint4*>(dst) = q;
  if (SPLIT) {
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    uint32_t r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      r[i] = pack_bf16x2(v[2 * i] - __uint_as_float(w[i] << 16), v[2 * i + 1] - __uint_as_float(w[i] & 0xFFFF0000u));
    *reinterpret_cast<uint4*>(dst + lo_off) = make_uint4(r[0], r[1], r[2], r[3]);
  }
}

__device__ __forceinline__ void bf16x8_to_float(const uint4& q, float* f) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}

// pre-encoded shared-memory descriptor halves (SWIZZLE_NONE): lo = start>>4 | (LBO>>4)<<16, hi = SBO>>4 | version 1
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16); }
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// conv GEMM of one row segment: D[seg rows][N] = sum_{k,s} A[rows + k][16-ch step s] * B_{k,s}
// a_lo already points at the segment's row 0; rows = buffer rows (chunk stride in 16-B units); b step = N*32 B.
// SPLIT: three MMAs per (tap, k-step) -- A_hi*B_hi + A_lo*B_hi + A_hi*B_lo (al16 / bl16 = distance of the low copies, 16-B units)
template <bool SPLIT>
__device__ __forceinline__ void issue_conv(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, int KS, int N,
                                           int rows, uint32_t idesc, uint32_t al16 = 0, uint32_t bl16 = 0) {
  uint32_t acc = 0;
#pragma unroll
  for (int k = 0; k < B2H_KW; ++k) {
    for (int s = 0; s < KS; ++s) {
      const uint32_t a = a_lo + 2 * s * rows + k, b = b_lo + (k * KS + s) * 2 * N;
      umma_bf16(d_tmem, desc64(a, a_hi), desc64(b, b_hi), idesc, acc);
      acc = 1;
      if (SPLIT) {
        umma_bf16(d_tmem, desc64(a + al16, a_hi), desc64(b, b_hi), idesc, 1);
        umma_bf16(d_tmem, desc64(a, a_hi), desc64(b + bl16, b_hi), idesc, 1);
      }
    }
  }
}

// Grid-wide barrier of a cooperative launch (all CTAs co-resident), flag form.  CTA c publishes the launch's token in
// flag[c] of the workspace header; warp 0 of every CTA polls all flags (one coalesced load per 32 CTAs): ONE L2 round trip
// after the last arrival (the arrival-counter form of round 1 needed three: atomicAdd, generation bump, poll).  The token
// is header[0] + 1, read by every CTA at kernel start and written back by CTA 0 after the barrier -- stale flags of
// earlier launches (any grid size) are always smaller.  Bounded spin: a protocol bug ends as a wrong answer + status.
__device__ __forceinline__ void grid_barrier_flags(unsigned* hdr, unsigned tok, int tid) {
  __syncthreads();
  volatile unsigned* flags = hdr + 4;
  if (tid == 0) {
    __threadfence();
    flags[blockIdx.x] = tok;
  }
  if (tid < 32) {
    const long long t0 = clock64();
    for (;;) {
      bool mine = true;
      for (int c = tid; c < (int)gridDim.x; c += 32) mine = mine && (flags[c] == tok);
      if (__all_sync(0xffffffffu, mine)) break;
      if (clock64() - t0 > 4000000000LL) {
        if (tid == 0) atomicExch(&g_tc_status, 50);
        break;
      }
    }
    __threadfence();
  }
  __syncthreads();
}

// torch.optim.Adam single-tensor update on one element whose state (m, v, p) was loaded earlier (before the grid barrier)
__device__ __forceinline__ void adam_apply(const FuseAdam& f, const Geo& g, const GpSlot& slot, int i, float gr, float m, float v,
                                           float p, float step_size, float inv_bc2_sqrt) {
  p = adam_update(m, v, p, gr * f.grad_scale, (float)(1.0 - f.beta1), (float)(1.0 - f.beta2), (float)f.beta2, f.eps, step_size,
                  inv_bc2_sqrt);
  f.m[i] = m; f.v[i] = v; f.params[i] = p;
  if (f.packed) scatter_packed(g, f.packed, slot, p);
}

#define B2H_STAMP() do { if (p.dbg && blockIdx.x == 0 && tid == 0 && dbg_n < 120) p.dbg[dbg_n++] = clock64(); } while (0)
// per-CTA wall-clock marks (ns, %globaltimer is common to all SMs): dbg[128 + 4 * cta + i], i = 0 start, 1 arrival at the
// grid barrier, 2 barrier passed, 3 end -- shows how much of a barrier wait is CTA launch skew
__device__ __forceinline__ long long global_ns() { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define B2H_MARK(i) do { if (p.dbg && tid == 0 && blockIdx.x < 192) p.dbg[128 + 4 * blockIdx.x + (i)] = global_ns(); } while (0)

// NT (128-row MMA tiles per segment) is a compile-time constant: with it at run time the per-row loops and the row
// context inside them cost the T <= 128 shapes ~6 % (27.4 -> 29.1 us per train step, 10.5 -> 11.3 us forward).
// SPLIT = fp32 mode: bf16 high/low operand pairs, three MMAs per product term group (see tile_smem_layout).
// VIEW (training only) = window views of frame streams: target / confidence rows through the view, per-window staging of
// the target tile.  A separate instantiation: the same code behind a run-time test made the dense 256x64 step 1.9 us
// slower (27.4 -> 29.3 us) with the same register count.  The forward kernel tests p.win_start at run time.
// UTT = sub-windows of utterances / training segments: window g reads its rows from the plan's table, rows at or past the
// sequence end are zero in every layer (the sequence ends there).  Forward (b2h_conv_forward_utterances): only the core rows
// are written, to y at their stream rows.  Training (b2h_train_*_utterances): target and confidence rows are read at the
// stream rows, the criterion covers the core rows with the weight 1 / (42 L_s) of the row's segment, the masked prediction
// goes to row (segment, frame in the segment) of y, and a plan the planning kernel refused ("bad") makes the step a no-op.
// CRIT (forward over utterances only) = validation over segments (b2h_validate_utterances): the layer-4 epilogue stores no
// prediction; it sums the criterion term |a s - t s| over the core rows of every sub-window against the target (and
// confidence) rows at the stream rows, and writes one sum per sub-window, reduced in a fixed order, to loss_partials[g].
template <bool TRAIN, int NT, bool SPLIT, bool VIEW = false, bool UTT = false, bool CRIT = false>
__global__ void __launch_bounds__(kTileThreads, 1) conv_tc_tile_kernel(TcTileArgs p) {
  static_assert(!(UTT && VIEW), "utterances and window views are separate instantiations");
  static_assert(!CRIT || (UTT && !TRAIN), "the validation criterion is a view of the forward over utterances");
  int dbg_n = 0;
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;      // MMAs of the current phase complete (one arrival per issuing warp)
  __shared__ __align__(8) uint64_t wbar;     // weights + biases landed (bulk async copies)
  __shared__ __align__(8) uint64_t tbar;     // target tile landed (train)
  __shared__ __align__(8) uint64_t ebar;     // backward: dZ_{l-1} stored and the dgrad accumulator read (one arrival per epilogue warp)
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float bias_s[4][64];
  __shared__ float red_s[8];
  __shared__ float crit_s[8][2];             // CRIT: per warp, per row segment: the sub-window's criterion sum
  const Geo& g = p.geo;
  const int T = p.T, MB = p.MB, HR = p.HR, nhalf = p.nhalf, gh = p.gh;
  constexpr int kWgCol = 64 * NT;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);     // warp-uniform
  const int rows = nhalf * HR;
  const int CH = rows * 16;
  const TileSmem L = tile_smem_layout(g, rows, TRAIN, SPLIT);
  const int LO = L.lo_off;                                       // byte distance of the low-half activation copies (SPLIT)
  const uint32_t al16 = (uint32_t)L.lo_off >> 4, bl16 = (uint32_t)L.wlo_off >> 4;
  unsigned char* G0 = smem + L.g0;
  unsigned char* G1 = smem + L.g1;
  unsigned char* X = smem + L.x;
  unsigned char* A1 = smem + L.a1;
  unsigned char* A2 = smem + L.a2;
  unsigned char* A3 = smem + L.a3;
  unsigned char* ONES = smem + L.ones;
  float* YS = reinterpret_cast<float*>(smem + L.ys);
  B2H_STAMP();   // kernel start
  if (TRAIN) B2H_MARK(0);

  // this thread's row: TMEM lane == tid & 127 (warps w and w+4 share lane quadrant w & 3 and split the columns)
  const int r128 = tid & 127;
  const int ch = warp >> 2;                      // column half: chunks c0 = 16*ch, 16*ch + 32, ...
  const int hh = (nhalf == 2) ? ((r128 >> 4) & 1) : 0;
  const int m = (nhalf == 2) ? ((r128 >> 5) * 16 + (r128 & 15)) : r128;
  // row context of this thread in MMA tile j of its segment (NT > 1 only with one 128*NT-row segment per tile)
  // UTT: us = the row's sub-window {stream row of frame 0, frame 0 in the utterance, clo | chi << 16, frames before the end}
  int utt_n = 0;                                 // UTT: sub-windows in the plan (read after griddep_wait)
  struct RowCtx { int row, t, gw; bool valid; int4 us; };
  auto rowctx = [&](int j, int wbase) {
    const int mm = m + 128 * j;
    const int wjj = mm / (T + 2);
    RowCtx r;
    r.t = mm - wjj * (T + 2);
    r.row = hh * HR + 2 + mm;
    r.gw = wbase + hh * gh + wjj;
    r.valid = (r.t < T) && (wjj < gh) && (r.gw < p.B);
    if constexpr (UTT) {
      const bool in = (wjj < gh) && (r.gw < utt_n);
      r.us = in ? __ldg(p.utt + 1 + r.gw) : make_int4(0, 0, 0, 0);
      r.valid = in && r.t < r.us.w;
    }
    return r;
  };
  const int wj = m / (T + 2), t = m - wj * (T + 2);     // tile 0 (prefetch path, NT == 1)
  const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
  const int srow = hh * MB + m;                  // row of this thread in the fp32 staging tile
  const bool bulk_io = (T & 1) == 0 && NT == 1 && !(SPLIT && TRAIN) && !UTT;  // T*168 B and the staging row offsets are 16-B multiples; the split training kernel has no staging tile; utterances write core rows only
  const int wpt = nhalf * gh;                    // windows per tile
  const int nissue = (nhalf == 2) ? 2 : NT;      // issuing warps: one per row segment / per 128-row MMA tile
  const uint32_t idesc_M = (nhalf == 2) ? 64 : 128;
  const int n_in = g.n_in;
  const bool vec_in = (g.pos_emb == 0) && ((n_in & 7) == 0) && n_in <= 32;   // <= 4 chunks: 16-B vector loads
  const bool fast_in = vec_in && NT == 1 && !UTT;   // + register prefetch one tile ahead
  const int seg_row = (nhalf == 2) ? HR : 128;   // row offset / TMEM offset of issuing warp w's accumulator
  const uint32_t seg_d = (nhalf == 2) ? (16u << 16) : 64u;
  const int cpr = n_in >> 3;

  // source row of (window gw, frame tt) in p.x; -1 = a zero row.  Dense batches: gw*T + tt.  Window views of a frame
  // stream: crop [start, start+T) cut at the clip end, then the pad rule (repeat the crop's first frame:
  // text_pose_dataset.py:511-518; zeros: :614-622) -- the same integer work as K0's windowing, bit-exact.
  // sub-window gw -> (window b, first frame, core rows [clo, chi)); identity when n_sub <= 1
  struct SubW { int b, start, clo, chi; };
  auto subw = [&](int gw) {
    SubW sw;
    if (p.n_sub <= 1) { sw.b = gw; sw.start = 0; sw.clo = 0; sw.chi = T; return sw; }
    sw.b = gw / p.n_sub;
    const SubWindow q = sub_window(p.T_orig, T, p.n_sub, gw - sw.b * p.n_sub);
    sw.start = q.start; sw.clo = q.clo; sw.chi = q.chi;
    return sw;
  };
  // row of (window gw, frame tt) in the dense (B, T, .) arrays (inputs, targets, scores, d_y, prediction)
  auto dense_row = [&](int gw, int tt) -> long long {
    if (p.n_sub <= 1) return (long long)gw * T + tt;
    const SubW sw = subw(gw);
    return (long long)sw.b * p.T_orig + sw.start + tt;
  };
  // row of (window / sub-window gw, frame tt) in p.x -- and in training also in p.target / p.conf
  auto xrow_of = [&](int gw, int tt) -> long long {
    if (!p.win_start) return dense_row(gw, tt);
    if (VIEW && p.n_sub > 1) {           // sub-window -> frame of its window's crop: context frames past win_end are pad
      const SubW sw = subw(gw);
      gw = sw.b; tt += sw.start;
    }
    const long long start = p.win_start[gw];
    long long cend = p.win_end ? p.win_end[gw] : p.n_frames;
    cend = cend > p.n_frames ? p.n_frames : cend;
    long long f = start + tt;
    if (f >= cend || f < 0) f = (p.pad_mode == B2H_PAD_REPEAT_FIRST && start >= 0 && start < cend) ? start : -1;
    return f;
  };
  // A viewed window's T target rows go to the staging tile as one bulk copy only when they are one contiguous run (the
  // crop is neither cut nor padded) starting at a 16-B aligned address: a row is 168 B, so odd stream rows sit 8 B off a
  // 16-B boundary (and the base pointer itself need only be 8-B aligned).  Other windows are staged row by row.
  auto view_bulk = [&](int gw) -> bool {
    const long long start = p.win_start[gw];
    long long cend = p.win_end ? p.win_end[gw] : p.n_frames;
    cend = cend > p.n_frames ? p.n_frames : cend;
    return start >= 0 && start + T <= cend && (reinterpret_cast<uintptr_t>(p.target + start * B2H_COUT) & 15) == 0;
  };
  // ---- input prefetch registers (one tile ahead) ----
  float4 xf[8];
  uint4 xb[4];
  auto load_x_row = [&](long long xr) {            // this thread's 16-B pieces of source row xr (zeros for xr < 0)
    if (p.x_dtype == B2H_DT_F32) {
      const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.x) + (size_t)(xr < 0 ? 0 : xr) * n_in);
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (c < 2 * cpr && ((c >> 1) & 1) == ch) xf[c] = xr < 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(src + c);
    } else {
      const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.x) + (size_t)(xr < 0 ? 0 : xr) * n_in);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < cpr && (c & 1) == ch) xb[c] = xr < 0 ? make_uint4(0, 0, 0, 0) : __ldg(src + c);
    }
  };
  auto prefetch_x = [&](int tile) {
    const int gw = tile * wpt + hh * gh + wj;
    const bool valid = (t < T) && (wj < gh) && (gw < p.B) && tile < p.n_tiles;
    if (!fast_in || !valid) return;
    load_x_row(xrow_of(gw, t));
  };
  // ---- part 1: nothing here reads or writes global memory, so under a programmatic dependent launch (launch_tc_tile)
  // it runs while the previous kernel of the stream is still in its tail ----
  griddep_launch_dependents();
  if (warp == 0) tmem_alloc(&tmem_slot, TRAIN ? 512 : 64 * NT);
  if (tid == 0) {
    mbar_init(&bar, nissue);
    mbar_init(&wbar, 1);
    mbar_init(&tbar, 1);
    if (TRAIN) mbar_init(&ebar, kTileThreads / 32 - 2);
    fence_barrier_init();
  }
  auto zero_buffers = [&]() {   // zero every activation / gradient buffer once: pad rows and pad channels stay zero
    const int act_bytes = L.ys;
    uint4* z = reinterpret_cast<uint4*>(smem);
    const uint4 zero = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < act_bytes / 16; i += kTileThreads) z[i] = zero;
  };
  // forward launches are programmatic: zero before the wait (under the predecessor); the train step is a normal launch
  // (the wait is then a no-op) and zeroes under its own loads in flight instead
  if (!TRAIN) zero_buffers();
  // ---- part 2: the previous kernel has completed and its writes (weights, Adam state, counters, inputs) are visible ----
  griddep_wait();
  B2H_STAMP();   // predecessor complete
  int utt_tiles = 0, utt_bad = 0;
  if constexpr (UTT) {                           // the plan's count: CTAs past it have no tile and load no weights
    utt_n = __ldg(&p.utt->x);
    if constexpr (TRAIN) utt_bad = __ldg(&p.utt->y);   // refused plan (count 0): no Adam update, no counter, NaN loss
    const int need = (utt_n + wpt - 1) / wpt;
    utt_tiles = need < p.n_tiles ? need : p.n_tiles;
  }
  prefetch_x(blockIdx.x);
  if (tid == 0 && (!UTT || (int)blockIdx.x < utt_tiles)) {
    // weights (packed bf16 UMMA blocks) + zero-padded biases -> smem once per CTA: 1-D bulk async copies (TMA engine)
    // that run under the first tile's input staging; completion is signalled on wbar.
    uint32_t total = 4 * 64 * 4;
    for (int l = 0; l < 4; ++l) {
      total += B2H_KW * g.kp[l] * g.np_[l] * 2 * (SPLIT ? 2 : 1);
      if (TRAIN && !SPLIT && l > 0) total += B2H_KW * round_up(g.cout[l], 16) * round_up(g.cin[l], 16) * 2;
    }
    mbar_arrive_expect_tx(&wbar, total);
    bulk_g2s(&bias_s[0][0], p.packed + g.bias_off, 4 * 64 * 4, &wbar);
    for (int l = 0; l < 4; ++l) {
      bulk_g2s(smem + L.wf[l], p.packed + g.tf_off[l], B2H_KW * g.kp[l] * g.np_[l] * 2, &wbar);
      if (SPLIT) bulk_g2s(smem + L.wf[l] + L.wlo_off, p.packed + g.tfl_off[l], B2H_KW * g.kp[l] * g.np_[l] * 2, &wbar);
      if (TRAIN && !SPLIT && l > 0)
        bulk_g2s(smem + L.wd[l], p.packed + g.td_off[l], B2H_KW * round_up(g.cout[l], 16) * round_up(g.cin[l], 16) * 2, &wbar);
    }
  }
  // Device-side counters.  Fused tail: every CTA reads the OLD values here (nobody writes them before the grid barrier,
  // which needs this CTA's arrival) and CTA 0 stores old + 1 after the barrier, so the bias corrections / the exchange
  // tag can be computed before the barrier.  Separate-launch paths: CTA 0 bumps them now for the kernels that follow.
  long long step_next = 0, epoch_next = 0;
  unsigned sync_tok = 0;
  int abort_flag = 0;
  if (TRAIN) {
    if (p.fuse.enabled) {
      step_next = *reinterpret_cast<const volatile long long*>(p.fuse.step_dev) + 1;
      if (p.fuse.world > 1) {
        epoch_next = *reinterpret_cast<const volatile long long*>(p.fuse.epoch_dev) + 1;
        abort_flag = *reinterpret_cast<volatile int*>(&g_dp_abort);
      }
      sync_tok = *reinterpret_cast<const volatile unsigned*>(p.fuse.hdr) + 1u;
    } else if (blockIdx.x == 0 && tid == 0 && !utt_bad) {
      if (p.step_dev) *p.step_dev += 1;
      if (p.epoch_dev) *p.epoch_dev += 1;
    }
  }
  if (TRAIN) zero_buffers();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;
  uint32_t phase = 0, tphase = 0, ephase = 0;
  float loss_acc = 0.0f;
  bool wg_started = false, weights_ready = false;
  B2H_STAMP();   // setup done

  // descriptor constants
  const uint32_t hi_k = desc_hi(128);            // K-major operands: SBO = 128 B (8-row groups contiguous)
  const uint32_t hi_mn = desc_hi((uint32_t)CH);  // MN-major operands: SBO = chunk stride
  const uint32_t acc_d = tbase + kAccCol;

  // Read one layer pair's weight / bias gradient accumulators out into this CTA's partial slice.  A pair shares its
  // TMEM columns: lanes 32q+i hold layer 2p (co = 16q+i), lanes 32q+16+i layer 2p+1, so one tcgen05.ld per tap
  // serves both layers and every lane has a row to store.  Column half 0 holds taps 0..2, half 1 taps 3..4 and the bias
  // column; the warp reads halves h0..h1 of its lane quadrant.
  auto readout_pair = [&](int pr, int h0, int h1) {
    float* part = p.partials + (size_t)blockIdx.x * gp_total(g);
    const int l = 2 * pr + (lane >> 4);
    const int co = (warp & 3) * 16 + (lane & 15);
    const bool mine = co < g.cout[l];
    const int Nw = g.kp[l];
    float* lp = part + gp_layer_off(g, l);
    float4* lp4 = reinterpret_cast<float4*>(lp);
    const int q4 = Nw >> 2, cout_l = g.cout[l];
    const uint32_t dcol = tbase + lane_addr + kWgCol + pr * kWgPairCols;
    for (int hc = h0; hc <= h1; ++hc) {
      const int k0 = hc == 0 ? 0 : 3, nk = hc == 0 ? 3 : 2;
      uint32_t v[3][32];
#pragma unroll
      for (int k = 0; k < 3; ++k)
        if (k < nk) tmem_ld32(dcol + (k0 + k) * 32, v[k]);
      uint32_t vb[16];
      if (hc == 1) tmem_ld16(dcol + 5 * 32, vb);      // 8 valid columns; column 0 holds db (ones sits in element 0)
      tmem_ld_wait();
      if (mine) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          if (k >= nk) continue;
          // slot layout [k][ci/4][co][4] (gp_slot_in_layer, b2h_common.cuh) as float4s: for a fixed (k, q) the 16 lanes
          // of a layer store 16 consecutive float4s
          float4* dst = lp4 + (size_t)(k0 + k) * q4 * cout_l + co;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (q * 4 < Nw)
              dst[(size_t)q * cout_l] = make_float4(__uint_as_float(v[k][4 * q]), __uint_as_float(v[k][4 * q + 1]),
                                                    __uint_as_float(v[k][4 * q + 2]), __uint_as_float(v[k][4 * q + 3]));
        }
        if (hc == 1) lp[B2H_KW * g.cout[l] * Nw + co] = __uint_as_float(vb[0]);
      }
    }
  };

  for (int tile = blockIdx.x; tile < (UTT ? utt_tiles : p.n_tiles); tile += gridDim.x) {
    const int wbase = tile * wpt;
    // sequence lengths of this thread's rows, fetched at tile start so the load is long complete at the layer-4 epilogue
    int lens[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const RowCtx rc = rowctx(j, wbase);
      const int Tw = p.n_sub > 1 ? p.T_orig : T;              // length of the window the sequence length refers to
      lens[j] = Tw;
      if (rc.valid && p.lengths) { const int v = p.lengths[p.n_sub > 1 ? rc.gw / p.n_sub : rc.gw]; lens[j] = v < 0 ? 0 : (v > Tw ? Tw : v); }
      if constexpr (UTT && TRAIN) if (rc.valid) lens[j] = __ldg(&p.utt_seg[rc.gw].y);   // the segment's length L_s
    }

    const bool tgt_smem = TRAIN && p.mode == 1 && bulk_io && p.n_sub <= 1;
    if (tid == 0) {
      if (!TRAIN) bulk_wait_read0();              // previous tile's y stores have read the staging tile
      if (tgt_smem) {                             // target rows of this tile's windows -> staging tile (TMA bulk loads)
        int nw = p.B - wbase; nw = nw > wpt ? wpt : nw;
        fence_proxy_async_smem();
        if (!VIEW) {
          mbar_arrive_expect_tx(&tbar, (uint32_t)nw * T * B2H_COUT * 4);
          for (int w = 0; w < nw; ++w) {
            const int h = w / gh, j = w - h * gh;
            bulk_g2s(YS + (size_t)(h * MB + j * (T + 2)) * B2H_COUT, p.target + (size_t)(wbase + w) * T * B2H_COUT,
                     (uint32_t)T * B2H_COUT * 4, &tbar);
          }
        } else {                                  // window views: the bulk-eligible windows only (view_bulk)
          int nb = 0;
          for (int w = 0; w < nw; ++w) nb += view_bulk(wbase + w) ? 1 : 0;
          mbar_arrive_expect_tx(&tbar, (uint32_t)nb * T * B2H_COUT * 4);
          for (int w = 0; w < nw; ++w) {
            if (!view_bulk(wbase + w)) continue;
            const int h = w / gh, j = w - h * gh;
            bulk_g2s(YS + (size_t)(h * MB + j * (T + 2)) * B2H_COUT, p.target + (size_t)p.win_start[wbase + w] * B2H_COUT,
                     (uint32_t)T * B2H_COUT * 4, &tbar);
          }
        }
      }
    }
    // ---- stage inputs: one thread per row (and per MMA tile j), (n_in) channels NWC -> X [chunk][row][8] bf16 ----
    for (int j = 0; j < NT; ++j) {
      const RowCtx rc = rowctx(j, wbase);
      const int row = rc.row;
      const int pe = g.pos_emb;
      const int nch0 = g.kp[0] / 8;
      if (rc.valid && vec_in) {
        if (!fast_in) load_x_row(UTT ? (long long)rc.us.x + rc.t : xrow_of(rc.gw, rc.t));   // no prefetch: load this row now
        if (p.x_dtype == B2H_DT_F32) {
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8)
            if (c8 < cpr && (c8 & 1) == ch) {
              const float4 lo = xf[2 * c8], hi = xf[2 * c8 + 1];
              const float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
              store8_act<SPLIT>(X, LO, CH, row, c8, v);
            }
        } else {
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8)
            if (c8 < cpr && (c8 & 1) == ch) {
              *reinterpret_cast<uint4*>(X + (size_t)c8 * CH + (size_t)row * 16) = xb[c8];
              if (SPLIT) *reinterpret_cast<uint4*>(X + LO + (size_t)c8 * CH + (size_t)row * 16) = make_uint4(0, 0, 0, 0);
            }
        }
      } else if (rc.valid) {
        const long long xr = UTT ? (long long)rc.us.x + rc.t : xrow_of(rc.gw, rc.t);
        for (int c8 = ch; c8 < nch0; c8 += 2) {
          float v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int cc = c8 * 8 + e;            // channel in the conv1 input (pos-emb row first)
            float val = 0.0f;
            if (pe && cc == 0) val = __fdiv_rn((float)((UTT ? rc.us.y : subw(rc.gw).start) + rc.t), (float)g.pe_len);   // HandPoseModels.py:70-82
            else if (cc - pe < n_in && cc - pe >= 0 && xr >= 0) {
              const size_t gi = (size_t)xr * n_in + (cc - pe);
              val = (p.x_dtype == B2H_DT_F32) ? __ldg(reinterpret_cast<const float*>(p.x) + gi)
                                              : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.x)[gi]);
            }
            v[e] = val;
          }
          store8_act<SPLIT>(X, LO, CH, row, c8, v);
        }
      } else {
        const uint4 zero = make_uint4(0, 0, 0, 0);
        for (int c8 = ch; c8 < nch0; c8 += 2) {
          *reinterpret_cast<uint4*>(X + (size_t)c8 * CH + (size_t)row * 16) = zero;
          if (SPLIT) *reinterpret_cast<uint4*>(X + LO + (size_t)c8 * CH + (size_t)row * 16) = zero;
        }
      }
      if (VIEW && tgt_smem && rc.valid && !view_bulk(rc.gw)) {
        // viewed window staged row by row: this thread's half of its row's 21 float2 (8-B aligned in any stream row), or
        // a zero row; read after the barrier below
        const long long tr = xrow_of(rc.gw, rc.t);
        const float2* src = reinterpret_cast<const float2*>(p.target + (tr < 0 ? 0 : tr) * B2H_COUT);
        float2* dst = reinterpret_cast<float2*>(YS + (size_t)srow * B2H_COUT);
        for (int q = ch * 11; q < (ch ? B2H_COUT / 2 : 11); ++q) dst[q] = tr < 0 ? make_float2(0.f, 0.f) : __ldg(src + q);
      }
      if (TRAIN && ch == 0) {   // ones column (B operand of the bias-gradient GEMM): 1 on real frames
        uint4 o = make_uint4(0, 0, 0, 0);
        if (rc.valid) o.x = 0x00003F80u;          // bf16(1.0) in element 0
        *reinterpret_cast<uint4*>(ONES + (size_t)row * 16) = o;
      }
    }
    prefetch_x(tile + gridDim.x);                 // next tile's rows travel while this tile computes
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    B2H_STAMP();   // staging done
    if (!weights_ready) { mbar_wait(&wbar, 0, 19); weights_ready = true; }
    B2H_STAMP();   // weights landed

    // =========================== forward: 4 conv layers ===========================
    for (int l = 0; l < 4; ++l) {
      unsigned char* bin = (l == 0) ? X : (l == 1) ? A1 : (l == 2) ? A2 : (TRAIN ? A3 : A1);
      unsigned char* bout = (l == 0) ? A1 : (l == 1) ? A2 : (TRAIN ? A3 : A1);
      const int KS = g.kp[l] >> 4, N = g.np_[l];
      if (warp < nissue) {
        if (elect_one()) {
          const uint32_t idesc = make_idesc_bf16(idesc_M, N, 0, 0);
          // output row 2+m of segment h reads input row m+k  ->  start row = h*HR + k
          const uint32_t a_lo = desc_lo(smem_u32(bin), (uint32_t)CH) + warp * seg_row;
          const uint32_t b_lo = desc_lo(smem_u32(smem + L.wf[l]), (uint32_t)N * 16);
          issue_conv<SPLIT>(acc_d + warp * seg_d, a_lo, hi_k, b_lo, hi_k, KS, N, rows, idesc, al16, bl16);
          umma_commit(&bar);
        }
        __syncwarp();
      }
      B2H_STAMP();   // fwd layer: MMAs issued
      mbar_wait(&bar, phase, 20 + l);
      phase ^= 1;
      tc_fence_after();
      B2H_STAMP();   // fwd layer: accumulator ready
      float contrib = 0.f;
#pragma unroll
      for (int j = 0; j < NT; ++j) {
      const RowCtx rc = rowctx(j, wbase);
      const int row = rc.row, t = rc.t, gw = rc.gw;
      const bool valid = rc.valid;
      const uint32_t taddr = tbase + lane_addr + kAccCol + 64 * j;
      if (l < 3) {
        for (int c0 = 16 * ch; c0 < N; c0 += 32) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
          float f[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) f[q] = valid ? fmaxf(__uint_as_float(v[q]) + bias_s[l][c0 + q], 0.0f) : 0.0f;
          store8_act<SPLIT>(bout, LO, CH, row, c0 >> 3, f);
          store8_act<SPLIT>(bout, LO, CH, row, (c0 >> 3) + 1, f + 8);
        }
      } else {
        // layer 4 epilogue: prediction (+ mask_output), and in train mode the criterion and d(loss)/d(pred)
        int len = lens[j];
        float n_el = 0.f, scale = 0.f;
        const float* tg = nullptr; const float* cf = nullptr; const float* dy = nullptr;
        // row of this frame in the dense (B, T, .) arrays; UTT: its stream row, written only in the sub-window's core
        const size_t drow = valid ? (UTT ? (size_t)rc.us.x + t : (size_t)dense_row(gw, t)) : 0;
        bool in_core = UTT ? (t >= (rc.us.z & 0xFFFF) && t < (rc.us.z >> 16)) : true, zrow = false;
        if (TRAIN && valid) {
          n_el = (float)len * (float)B2H_COUT;                      // (sub-window mode: len = the WINDOW's sequence length)
          scale = (p.loss_kind == B2H_LOSS_L1) ? (1.0f / (float)p.loss_B) / n_el : 1.0f / n_el;
          if (p.n_sub > 1) {                                        // criterion on the core rows only; len -> sub-window frames
            const SubW sw = subw(gw);
            in_core = t >= sw.clo && t < sw.chi;
            len -= sw.start;
          }
          if (p.mode == 1) {                                        // global copy (used when the tile is not staged)
            long long trow = (long long)drow;
            if (VIEW) {                                             // window view: the stream row; a zero row reads as zeros
              trow = xrow_of(gw, t);
              zrow = trow < 0;
              trow = zrow ? 0 : trow;
            }
            tg = p.target + trow * B2H_COUT;
            cf = p.conf ? p.conf + trow * (B2H_COUT / 2) : nullptr;
          } else {
            dy = p.d_y + drow * B2H_COUT;
          }
        }
        const bool y_smem = !TRAIN && bulk_io;
        size_t prow = drow;                                         // training over segments: (segment, frame in it)
        if constexpr (UTT && TRAIN) prow = valid ? (size_t)__ldg(&p.utt_seg[gw].x) * p.utt_max_len + rc.us.y + t : 0;
        float* yrow = (valid && p.y && in_core) ? p.y + prow * B2H_COUT : nullptr;                // global row
        float* ys_row = YS + (size_t)srow * B2H_COUT;                                            // shared staging row
        if (tgt_smem && j == 0) { mbar_wait(&tbar, tphase, 18); tphase ^= 1; }
        B2H_STAMP();   // layer-4 epilogue: target tile landed
        float sum = 0.f;
        // Fast path of the headline configuration (maskedPoseL1 inside, target tile staged in shared memory, prediction
        // not requested): the chunk's first column is a compile-time constant, so every `column < 42` test folds away
        // and the body is straight-line code -- the generic loop below executed ~4x the instructions of a hidden
        // layer's epilogue (per-element predicates for the confidence weights, the given-d_y mode and the y store).
        const bool l4_fast = TRAIN && p.mode == 1 && p.loss_kind == B2H_LOSS_L1 && tgt_smem && p.y == nullptr;
        if constexpr (CRIT) {
          // validation: the criterion term of the training epilogue (L1 = the weighted form with s = 1) on the core rows
          // before the segment end; target rows are 168 B, 8-B aligned at odd stream rows: float2 loads
          const bool live = valid && in_core;
          const float* trow = p.target + (live ? drow : 0) * B2H_COUT;
          const float* crow = (p.loss_kind == B2H_LOSS_CONFL1) ? p.conf + (live ? drow : 0) * (B2H_COUT / 2) : nullptr;
          for (int c0 = 16 * ch; c0 < N; c0 += 32) {
            uint32_t v[16];
            tmem_ld16(taddr + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 16; q += 2) {
              const int c = c0 + q;
              if (live && c < B2H_COUT) {
                const float2 tv = __ldg(reinterpret_cast<const float2*>(trow + c));
                const float sv = crow ? __ldg(crow + (c >> 1)) : 1.0f;
                const float a0 = __uint_as_float(v[q]) + bias_s[3][c], a1 = __uint_as_float(v[q + 1]) + bias_s[3][c + 1];
                sum += fabsf(__fsub_rn(__fmul_rn(a0, sv), __fmul_rn(tv.x, sv)));
                sum += fabsf(__fsub_rn(__fmul_rn(a1, sv), __fmul_rn(tv.y, sv)));
              }
            }
          }
          contrib += sum;
        } else if (TRAIN && l4_fast) {
          const bool live = valid && (t < len) && in_core;   // rows t >= len are zeroed by mask_output and carry no loss
          auto chunk = [&](auto c0_tag) {
            constexpr int C0 = decltype(c0_tag)::value;
            uint32_t v[16];
            tmem_ld16(taddr + C0, v);
            float tv[16];
            const float2* tp = reinterpret_cast<const float2*>(ys_row + C0);
#pragma unroll
            for (int q2 = 0; q2 < 8; ++q2) {
              if (C0 + 2 * q2 < B2H_COUT) { const float2 t2 = tp[q2]; tv[2 * q2] = t2.x; tv[2 * q2 + 1] = t2.y; }
              else { tv[2 * q2] = 0.f; tv[2 * q2 + 1] = 0.f; }
            }
            tmem_ld_wait();
            float gq[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              if (C0 + q < B2H_COUT) {
                const float a = live ? __uint_as_float(v[q]) + bias_s[3][C0 + q] : 0.0f;      // masked prediction
                const float d = __fsub_rn(a, tv[q]);        // == a*1 - t*1 of the weighted form, exactly
                sum += live ? fabsf(d) : 0.0f;
                const float gr = d > 0.f ? scale : (d < 0.f ? -scale : 0.f);
                gq[q] = live ? gr : 0.0f;
              } else {
                gq[q] = 0.0f;
              }
            }
            store8_act<SPLIT>(G0, LO, CH, row, C0 >> 3, gq);
            store8_act<SPLIT>(G0, LO, CH, row, (C0 >> 3) + 1, gq + 8);
          };
          if (ch == 0) { chunk(std::integral_constant<int, 0>{}); chunk(std::integral_constant<int, 32>{}); }
          else chunk(std::integral_constant<int, 16>{});
          B2H_STAMP();   // layer-4 epilogue: chunks done (fast path)
          B2H_STAMP();
        } else
        for (int c0 = 16 * ch; c0 < N; c0 += 32) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
          float gq[16];
          if (!TRAIN) {
            // inference epilogue: bias, optional mask_output (utils.py:309-312) / de-normalise, store the row
            const bool masked = p.apply_mask && (t >= len);
#pragma unroll
            for (int q = 0; q < 16; q += 2) {
              const int c = c0 + q;
              if (yrow && c < B2H_COUT) {
                float a = __uint_as_float(v[q]) + bias_s[3][c];
                float b = __uint_as_float(v[q + 1]) + bias_s[3][c + 1];
                if (masked) { a = 0.0f; b = 0.0f; }
                else if (p.out_scale != 1.0f) { a *= p.out_scale; b *= p.out_scale; }
                if (y_smem) *reinterpret_cast<float2*>(ys_row + c) = make_float2(a, b);
                else *reinterpret_cast<float2*>(yrow + c) = make_float2(a, b);
              }
            }
          } else {
            // training epilogue, branch-free per element: masked prediction, criterion term, d(loss)/d(pred).
            // L1 is the confidence-weighted form with s = 1 (a*1 - t*1 == a - t exactly).   utils.py:422-426 / :447-450
            const bool live = valid && (t < len) && in_core;   // rows t >= len are zeroed by mask_output and carry no loss
            float tvals[16], svals[16];
#pragma unroll
            for (int q = 0; q < 16; q += 2) {
              float2 tv2 = make_float2(0.f, 0.f);
              float sv = 1.0f;
              if (live && c0 + q < B2H_COUT) {
                if (p.mode == 1) tv2 = tgt_smem ? *reinterpret_cast<const float2*>(ys_row + c0 + q) : __ldg(reinterpret_cast<const float2*>(tg + c0 + q));
                else tv2 = __ldg(reinterpret_cast<const float2*>(dy + c0 + q));
                if (cf && p.loss_kind == B2H_LOSS_CONFL1) sv = __ldg(cf + ((c0 + q) >> 1));
                if (VIEW && zrow) { tv2 = make_float2(0.f, 0.f); sv = (cf && p.loss_kind == B2H_LOSS_CONFL1) ? 0.f : 1.0f; }
              }
              tvals[q] = tv2.x; tvals[q + 1] = tv2.y; svals[q] = sv; svals[q + 1] = sv;
            }
            const bool given_dy = (p.mode != 1);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const int c = c0 + q;
              const bool on = live && (c < B2H_COUT);
              const float a = on ? __uint_as_float(v[q]) + bias_s[3][c < 64 ? c : 63] : 0.0f;      // masked prediction
              const float sv = svals[q];
              const float d = __fsub_rn(__fmul_rn(a, sv), __fmul_rn(tvals[q], sv));
              sum += on ? fabsf(d) : 0.0f;
              const float sc = sv * scale;
              float gr = d > 0.f ? sc : (d < 0.f ? -sc : 0.f);
              gr = given_dy ? tvals[q] : gr;                // backward of a given d_y: the staged value IS the gradient
              gq[q] = on ? gr : 0.0f;
              if (yrow && c < B2H_COUT && valid) yrow[c] = a;
            }
          }
          if (TRAIN) {
            store8_act<SPLIT>(G0, LO, CH, row, c0 >> 3, gq);
            store8_act<SPLIT>(G0, LO, CH, row, (c0 >> 3) + 1, gq + 8);
          }
          B2H_STAMP();   // layer-4 epilogue: one 16-column chunk done
        }
        // per-sample mean = sum_{t<len} |d| / (len*42)  (utils.py:426 / :450): accumulate sum/n_el
        if (TRAIN && p.mode == 1) contrib += (valid && t < len && in_core) ? sum / n_el : 0.f;
      }
      }   // MMA tiles j
      if (TRAIN && p.mode == 1 && l == 3) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        if (lane == 0) red_s[warp] = contrib;
      }
      if constexpr (CRIT) if (l == 3) {
        // lanes 0-15 / 16-31 of a warp hold rows of row segment 0 / 1 when a tile holds two (nhalf == 2)
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        if ((lane & 15) == 0) crit_s[warp][lane >> 4] = contrib;
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncthreads();
      tc_fence_after();
      if (!TRAIN && l == 3 && bulk_io && tid == 0 && p.y) {   // y tile -> global: one TMA bulk store per window
        int nw = p.B - wbase; nw = nw > wpt ? wpt : nw;
        for (int w = 0; w < nw; ++w) {
          const int h = w / gh, j = w - h * gh;
          bulk_s2g(p.y + (size_t)(wbase + w) * T * B2H_COUT, YS + (size_t)(h * MB + j * (T + 2)) * B2H_COUT, (uint32_t)T * B2H_COUT * 4);
        }
        bulk_commit();
      }
      if constexpr (CRIT) if (l == 3 && tid < nhalf) {   // one sub-window per row segment (gh == 1: Ts >= 64, launch_tc_tile)
        float s = 0.f;
        for (int w = 0; w < 8; ++w) s += nhalf == 2 ? crit_s[w][tid] : crit_s[w][0] + crit_s[w][1];
        if (wbase + tid < utt_n) p.loss_partials[wbase + tid] = s;
      }
      B2H_STAMP();   // fwd layer: epilogue done
    }
    if (TRAIN && p.mode == 1 && tid == 0) loss_acc += ((red_s[0] + red_s[1]) + (red_s[2] + red_s[3])) + ((red_s[4] + red_s[5]) + (red_s[6] + red_s[7]));

    if (TRAIN) {
      // =========================== backward ===========================
      // dZ_l (grad wrt layer l's pre-activation) ping-pongs G0 (l=3) -> G1 (l=2) -> G0 (l=1) -> G1 (l=0).
      // Warps 0/1 only issue: the tensor pipe runs D4 W4 D3 W3 D2 W2 W1 back to back, and the issuers wait only for the
      // epilogue handshake (ebar) before each dgrad and for each other between dgrad and wgrad.  Warps 2..7 wait for dgrad_l's commit and run its ReLU-mask
      // epilogue while wgrad_l is in the pipe; warps 4/5 take all columns of lane quadrants 0/1.  The epilogue's only
      // write hazard, the dZ buffer wgrad_{l+1} read, is clear: that commit also covers wgrad_{l+1}.
      const bool last_tile = tile + (int)gridDim.x >= (UTT ? utt_tiles : p.n_tiles);
      const bool both = warp == 4 || warp == 5;
      for (int l = 3; l >= 0; --l) {
        unsigned char* gz = ((3 - l) & 1) ? G1 : G0;          // dZ_l
        unsigned char* gnext = ((3 - l) & 1) ? G0 : G1;       // dZ_{l-1}
        unsigned char* ain = (l == 0) ? X : (l == 1) ? A1 : (l == 2) ? A2 : A3;   // layer l's input activation
        if (warp < nissue) {
          if (elect_one()) {
            if (l < 3) {                         // dZ_l is in shared memory and the dgrad accumulator has been read
              mbar_wait(&ebar, ephase, 40 + l);
              tc_fence_after();
              B2H_STAMP();   // bwd layer: epilogue handshake passed
            }
            if (l > 0) {  // dgrad: dA_{l-1}[r][ci] = sum_{k',co} dZ_l[r+k'-2][co] * W_l[co][ci][4-k']
              const int KSd = round_up(g.cout[l], 16) >> 4, Nd = round_up(g.cin[l], 16);
              const uint32_t a_lo = desc_lo(smem_u32(gz), (uint32_t)CH) + warp * seg_row;
              if (!SPLIT) {
                const uint32_t idesc = make_idesc_bf16(idesc_M, Nd, 0, 0);
                const uint32_t b_lo = desc_lo(smem_u32(smem + L.wd[l]), (uint32_t)Nd * 16);
                issue_conv<false>(acc_d + warp * seg_d, a_lo, hi_k, b_lo, hi_k, KSd, Nd, rows, idesc);
              } else {
                // No transposed weight blocks in split mode: the FORWARD blocks [tap][ci/8][co row][8 ci] are read as an
                // MN-major B operand (N = ci: 8-element groups np*16 B apart = SBO; K = co: rows of 16 B, 8-row groups 128 B
                // apart = LBO), tap k' of the dgrad = forward tap 4-k', K-step s' = co rows 16 s' ..
                const uint32_t idesc = make_idesc_bf16(idesc_M, Nd, 0, 1);
                const int KSf = g.kp[l] >> 4, Nf = g.np_[l];
                const uint32_t hi_w = desc_hi((uint32_t)Nf * 16);
                const uint32_t b0 = desc_lo(smem_u32(smem + L.wf[l]), 128);
                uint32_t acc = 0;
#pragma unroll
                for (int k = 0; k < B2H_KW; ++k)
                  for (int sd = 0; sd < KSd; ++sd) {
                    const uint32_t a = a_lo + 2 * sd * rows + k;
                    const uint32_t b = b0 + (uint32_t)((B2H_KW - 1 - k) * KSf * Nf * 2 + 16 * sd);
                    const uint32_t d = acc_d + warp * seg_d;
                    umma_bf16(d, desc64(a, hi_k), desc64(b, hi_w), idesc, acc);
                    acc = 1;
                    umma_bf16(d, desc64(a + al16, hi_k), desc64(b, hi_w), idesc, 1);
                    umma_bf16(d, desc64(a, hi_k), desc64(b + bl16, hi_w), idesc, 1);
                  }
              }
              umma_commit(&bar);
            }
          }
          __syncwarp();
          // both segments' dgrad enter the tensor pipe ahead of either warp's wgrad, so that the epilogue can start as
          // soon as possible
          if (nissue == 2 && l > 0) named_bar_sync(1, 64);
          if (elect_one()) {
            // wgrad: dW_l[k][co][ci] += sum_r dZ_l[r][co] * in_l[r+k-2][ci];  db_l[co] += sum_r dZ_l[r][co]
            // A = dZ_l read MN-major (M = co, 8 chunks), B = in_l read MN-major (N = ci), K = 16 frames per MMA.
            // The six accumulators (5 taps + bias) are split between the issuing warps (disjoint TMEM columns).
            {
              const int Nw = g.kp[l];
              const uint32_t idw = make_idesc_bf16(64, Nw, 1, 1), idb = make_idesc_bf16(64, 8, 1, 1);
              const uint32_t a_lo0 = desc_lo(smem_u32(gz), 128), b_lo0 = desc_lo(smem_u32(ain), 128), o_lo0 = desc_lo(smem_u32(ONES), 128);
              const uint32_t dcol = tbase + kWgCol + (l >> 1) * kWgPairCols + ((uint32_t)((l & 1) * 16) << 16);
              for (int h = 0; h < nhalf; ++h)
                for (int s = 0; s < MB / 16; ++s) {
                  const uint32_t first = (h == 0 && s == 0 && !wg_started) ? 0u : 1u;
                  const uint32_t r0 = h * HR + 2 + 16 * s;           // rows (16-B units)
                  const uint64_t ad = desc64(a_lo0 + r0, hi_mn);
#pragma unroll
                  for (int k = 0; k < B2H_KW + 1; ++k) {
                    if (nissue == 2 && (k & 1) != warp) continue;
                    if (k < B2H_KW) {
                      const uint64_t bd = desc64(b_lo0 + r0 + k - 2, hi_mn);
                      umma_bf16(dcol + k * 32, ad, bd, idw, first);
                      if (SPLIT) {      // dZ_lo * in_hi + dZ_hi * in_lo
                        umma_bf16(dcol + k * 32, desc64(a_lo0 + r0 + al16, hi_mn), bd, idw, 1);
                        umma_bf16(dcol + k * 32, ad, desc64(b_lo0 + r0 + k - 2 + al16, hi_mn), idw, 1);
                      }
                    } else {
                      umma_bf16(dcol + 5 * 32, ad, desc64(o_lo0 + r0, hi_mn), idb, first);
                      if (SPLIT) umma_bf16(dcol + 5 * 32, desc64(a_lo0 + r0 + al16, hi_mn), desc64(o_lo0 + r0, hi_mn), idb, 1);
                    }
                  }
                }
              if (l == 0) umma_commit(&bar);     // last MMAs of the tile: fence the buffers before restaging
            }
          }
          __syncwarp();
        }
        if (warp < 2) {                          // (warp 1 idles when one warp issues: nissue == 1)
          if (l < 3) ephase ^= 1;
          if (l > 0) phase ^= 1;                 // the issuers do not wait for the dgrad commits
          B2H_STAMP();   // bwd layer: MMAs issued
        } else if (l > 0) {
          mbar_wait_warp(&bar, phase, 30 + l);   // dgrad_l complete (and with it wgrad_{l+1}, issued before it)
          phase ^= 1;
          tc_fence_after();
          // dZ_{l-1} = dA_{l-1} * (a_{l-1} > 0)     (ReLU backward on the saved activation)
          const int Nd = round_up(g.cin[l], 16);
          for (int j = 0; j < NT; ++j) {
          const RowCtx rc = rowctx(j, wbase);
          const int row = rc.row;
          const bool valid = rc.valid;
          const uint32_t taddr = tbase + lane_addr + kAccCol + 64 * j;
          for (int c0 = both ? 0 : 16 * ch; c0 < Nd; c0 += both ? 16 : 32) {
            uint32_t v[16];
            tmem_ld16(taddr + c0, v);
            tmem_ld_wait();
            float f[16], act[16];
            bf16x8_to_float(*reinterpret_cast<const uint4*>(ain + (size_t)(c0 >> 3) * CH + (size_t)row * 16), act);
            bf16x8_to_float(*reinterpret_cast<const uint4*>(ain + (size_t)((c0 >> 3) + 1) * CH + (size_t)row * 16), act + 8);
#pragma unroll
            for (int q = 0; q < 16; ++q) f[q] = (valid && act[q] > 0.0f) ? __uint_as_float(v[q]) : 0.0f;
            store8_act<SPLIT>(gnext, LO, CH, row, c0 >> 3, f);
            store8_act<SPLIT>(gnext, LO, CH, row, (c0 >> 3) + 1, f + 8);
          }
          }   // MMA tiles j
          // hand dZ_{l-1} (generic-proxy stores) and the free dgrad accumulator to the issuers
          fence_proxy_async_smem();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&ebar);
          if (l == 1 && last_tile) {
            // last tile of this CTA: W_4 and W_3 (layer pair 1) are final (their MMAs precede dgrad_1's commit) -> read
            // them out under the tensor-pipe time of W_2 / W_1
            readout_pair(1, both ? 0 : ch, both ? 1 : ch);
          }
        }
      }
      mbar_wait(&bar, phase, 30);                // wgrad_0: every MMA of the tile is complete
      phase ^= 1;
      B2H_STAMP();   // bwd: last weight-gradient MMA complete
      fence_proxy_async_smem();
      tc_fence_before();
      __syncthreads();
      tc_fence_after();
      B2H_STAMP();   // bwd: epilogue warps done (pair-1 read-out)
      wg_started = true;
    }
  }

  if (TRAIN) {
    // ---- read the remaining weight / bias gradient accumulators out into this CTA's partial slice ----
    if (!wg_started) {
      float* part = p.partials + (size_t)blockIdx.x * gp_total(g);
      for (int i = tid; i < gp_total(g); i += kTileThreads) part[i] = 0.0f;
    } else {
      readout_pair(0, ch, ch);                     // (pair 1 was read out under the last tile's W2 / W1)
    }
    if (tid == 0 && p.loss_partials) {
      float lp = (p.loss_kind == B2H_LOSS_L1) ? loss_acc / (float)p.loss_B : loss_acc;
      if constexpr (UTT) if (utt_bad) lp = __int_as_float(0x7fffffff);   // a refused segment list: the loss is NaN
      p.loss_partials[blockIdx.x] = lp;
    }
    B2H_STAMP();   // partial slice written

    if (p.fuse.enabled) {
      // ===== same launch: cross-CTA reduction (+ peer exchange) + Adam + weight re-pack =====
      const FuseAdam& f = p.fuse;
      __shared__ float s_step_size, s_inv_bc2_sqrt;
      const int nj = gp_total(g);                        // multiple of 4: every slice is float4-addressable
      const int nparts = (int)gridDim.x;
      const int per = round_up((nj + nparts - 1) / nparts, 4);
      const int j0 = (int)blockIdx.x * per;
      const int j_end = min(nj, j0 + per);
      const bool dp = f.world > 1;
      // ---- work that does not need the other CTAs, done while the slowest CTA is still on its way to the barrier:
      // bias corrections (double-precision powers), decode of this thread's slot, its Adam state (m, v, p) ----
      if (tid == kTileThreads - 1) {                     // last thread: usually idle in the gather below
        // bias corrections 1 - beta^t = -expm1(t * log1p(beta - 1)) in fp32 (relative error ~3e-7 for every t, also
        // where 1 - beta^t cancels): the double-precision powers of round 1 cost ~5k cycles on B200's few FP64 units
        const float lr = (float)(f.lr_dev ? *f.lr_dev : f.lr);
        const float tt = (float)step_next;
        const float bc1 = -expm1f(tt * log1pf((float)(f.beta1 - 1.0)));
        const float bc2 = -expm1f(tt * log1pf((float)(f.beta2 - 1.0)));
        s_step_size = lr / bc1;
        s_inv_bc2_sqrt = 1.0f / sqrtf(bc2);
      }
      const bool one_pass = per <= kTileThreads;         // the usual case: one slot per thread
      GpSlot my_slot;
      int my_i = -1;
      float my_m = 0.f, my_v = 0.f, my_p = 0.f;
      if (one_pass && j0 + tid < j_end && gp_decode(g, j0 + tid, my_slot)) {
        my_i = gp_flat_of_slot(g, my_slot);
        my_m = __ldcg(f.m + my_i); my_v = __ldcg(f.v + my_i); my_p = __ldcg(f.params + my_i);
      }
      B2H_MARK(1);
      bool aborted = abort_flag != 0;                    // set by an earlier step's peer timeout (fetched at kernel start)
      grid_barrier_flags(f.hdr, sync_tok, tid);          // every CTA's partial slice is visible
      B2H_STAMP();   // tail: grid barrier passed
      B2H_MARK(2);
      if (blockIdx.x == 0 && tid == 0) {                 // publish the counters for the next launch
        *reinterpret_cast<volatile unsigned*>(f.hdr) = sync_tok;
        if (!utt_bad) *p.step_dev = step_next;
        if (dp) *p.epoch_dev = epoch_next;
      }
      if (blockIdx.x == 0 && warp == 7 && f.loss_out) {  // loss = sum of the CTAs' loss partials (fixed order)
        float sl = 0.f;
        for (int c = lane; c < (int)gridDim.x; c += 32) sl += __ldcg(p.loss_partials + c);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sl += __shfl_xor_sync(0xffffffffu, sl, o);
        if (lane == 0) *f.loss_out = sl;
      }
      // Data-parallel exchange buffer (per rank, peer-mapped): 32-bit words [2 (epoch parity)][world (source rank)][nj].
      // A word is either the SENTINEL (a NaN pattern no arithmetic produces) or a peer's fp32 gradient slot: the value is its
      // own arrival flag, so a slot costs 4 bytes on the wire (round 1's {value, epoch tag} words cost 8: at 8 ranks the
      // 1.36 MB of ingress per step were ~1.5 us of NVLink time).  The reader puts the sentinel back right after reading;
      // the parity double-buffers against a peer that is one step ahead (it cannot be two ahead: it needs this rank's words
      // of the step in between, which are pushed by the NEXT launch, after this launch's resets are complete).
      const long long epoch = epoch_next;
      const size_t ll_src = ((size_t)(epoch & 1) * f.world + f.rank) * nj;
      // Latency-bound L2 gather of this CTA's `per` slots over all CTA slices: float4 columns x part groups, 16
      // independent 16-B loads in flight per thread, fixed summation order (deterministic).
      // [groups][ncol] partial sums: the staging tile is free now (split training kernel: the activation buffers are --
      // every MMA that read them has completed)
      float4* red4 = reinterpret_cast<float4*>(L.has_ys ? smem + L.ys : smem);
      for (int jb = j0; jb < j_end; jb += 4096) {        // <= 1024 float4 columns (16 KB of staging) per pass
        const int jn = min(j_end, jb + 4096);
        const int ncol = (jn - jb + 3) >> 2;
        int groups = kTileThreads / ncol; groups = groups < 1 ? 1 : (groups > 8 ? 8 : groups);
        const int cpg = kTileThreads / groups;            // columns handled per sweep
        for (int cb = 0; cb < ncol; cb += cpg) {
          const int col = cb + tid % cpg, pg = tid / cpg;
          if (col < ncol && pg < groups) {
            const float4* src = reinterpret_cast<const float4*>(p.partials + jb + 4 * col);
            const size_t stride4 = (size_t)nj >> 2;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int c = pg; c < nparts; c += kGatherDepth * groups) {
              float4 v[kGatherDepth];                     // 128 slices / 6 groups = 22 loads: one batch in flight
#pragma unroll
              for (int u = 0; u < kGatherDepth; ++u) {
                const int cc = c + u * groups;
                v[u] = (cc < nparts) ? __ldcg(src + (size_t)cc * stride4) : make_float4(0.f, 0.f, 0.f, 0.f);
              }
#pragma unroll
              for (int u = 0; u < kGatherDepth; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
            }
            red4[pg * ncol + col] = acc;
          }
        }
        __syncthreads();
        B2H_STAMP();   // tail: gather done
        const float* red = reinterpret_cast<const float*>(red4);
        for (int j = jb + tid; j < jn; j += kTileThreads) {
          float gr = 0.f;
          for (int pg = 0; pg < groups; ++pg) gr += red[(size_t)pg * ncol * 4 + (j - jb)];
          bool apply = !utt_bad;                         // a refused segment list leaves params, m, v and packed as they are
          // padding slots of the slot layout (ci >= cin, bias pad: ~10 % at C = 30) carry no parameter: neither pushed nor polled
          const bool real_slot = one_pass ? (my_i >= 0) : (flat_index_of_gp(g, j) >= 0);
          if (dp && real_slot) {
            // push my slot to every rank, then collect the world's slots for the same j from my own buffer and sum them
            // in rank order (identical arithmetic on every rank).  With a multicast (NVLS) mapping of the exchange
            // buffers ONE multimem.st is replicated by the NVSwitch into every rank's buffer; otherwise W unicast
            // 4-byte stores (coalesced per warp, fire-and-forget over NVLink).  The word is its own arrival flag: the
            // reader's buffer holds the sentinel until the value lands, and the reader re-arms it after use.
            uint32_t word = __float_as_uint(gr);
            if (word == kDpSentinel) word = 0x7FC00000u;               // (a NaN gradient stays a NaN, never the sentinel)
            if (f.mc_buf) {
              asm volatile("multimem.st.relaxed.sys.global.b32 [%0], %1;" ::"l"(reinterpret_cast<uint32_t*>(f.mc_buf) + ll_src + j), "r"(word) : "memory");
            } else {
              for (int r = 0; r < f.world; ++r)
                *(reinterpret_cast<volatile uint32_t*>(const_cast<float*>(f.peer_bufs[r])) + ll_src + j) = word;
            }
            B2H_STAMP();   // tail: slot pushed
            float gsum = 0.f;
            volatile uint32_t* mine = reinterpret_cast<volatile uint32_t*>(const_cast<float*>(f.peer_bufs[f.rank])) + (size_t)(epoch & 1) * f.world * nj + j;
            const long long t0 = clock64();
            for (int rb = 0; rb < f.world; rb += 8) {
              // All (<= 8) ranks' words are requested together and the whole group is re-read until every one has arrived:
              // one L2 round trip per polling round.  (Round 1 re-polled the missing words one after the other -- at 8
              // ranks the first read comes back stale for almost everyone, which cost one round trip PER RANK.)
              uint32_t w[8];
              bool all_here;
              do {
#pragma unroll
                for (int u = 0; u < 8; ++u)
                  if (rb + u < f.world) w[u] = mine[(size_t)(rb + u) * nj];
                all_here = true;
#pragma unroll
                for (int u = 0; u < 8; ++u)
                  if (rb + u < f.world) all_here = all_here && (w[u] != kDpSentinel);
                if (!all_here && clock64() - t0 > 6000000000LL) {        // ~3 s: a peer never arrived
                  atomicExch(&g_tc_status, 51);
                  atomicExch(&g_dp_abort, 1);
                  aborted = true;
                  break;
                }
              } while (!all_here);
#pragma unroll
              for (int u = 0; u < 8; ++u)
                if (rb + u < f.world) {
                  gsum += __uint_as_float(w[u]);                       // rank order: identical arithmetic on every rank
                  if (!aborted) mine[(size_t)(rb + u) * nj] = kDpSentinel;   // re-arm the word for the step after next
                }
            }
            B2H_STAMP();   // tail: world's slots collected
            gr = gsum;
            // Sticky abort: after a peer timeout no parameter / moment is written by the threads that missed a word, nor
            // by anybody in any later step, until the host has read and cleared the status (the flag of earlier steps
            // was fetched before the grid barrier) -- replicas may stall, the failure is never silent.
            apply = !aborted;
          }
          if (apply) {
            if (one_pass) {
              if (my_i >= 0) adam_apply(f, g, my_slot, my_i, gr, my_m, my_v, my_p, s_step_size, s_inv_bc2_sqrt);
            } else {
              GpSlot sl;
              if (gp_decode(g, j, sl)) {
                const int i = gp_flat_of_slot(g, sl);
                adam_apply(f, g, sl, i, gr, f.m[i], f.v[i], f.params[i], s_step_size, s_inv_bc2_sqrt);
              }
            }
          }
        }
        __syncthreads();
      }
      B2H_STAMP();   // tail: reduction (+ exchange) + Adam done
      B2H_MARK(3);
    }
  }
  if (!TRAIN && tid == 0) bulk_wait0();
  B2H_STAMP();   // readout done
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, TRAIN ? 512 : 64 * NT);
}

// ---- host side ----
// Training of windows longer than one tile segment (128 frames in fp32 mode, 256 in bf16 mode): n_sub overlapping
// sub-windows of Ts frames (see TcTileArgs), every cut with >= 16 real frames of context on both sides: the two edge
// sub-windows carry up to Ts - 16 core frames, the interior ones Ts - 32.
constexpr int kTileMaxTrainT = 4096;

TilePlan plan_tile(const Geo& g, int B, int T, bool train, bool split) {
  TilePlan p{};
  p.train = train; p.split = split;
  if (T < 1 || T > (train ? kTileMaxTrainT : 256)) return p;
  if ((g.kp[0] > 32 || g.kp[1] > 32) && (train || split || g.kp[0] > 64 || g.kp[1] > 64)) return p;
  p.n_sub = 1;
  const int Ts = split ? 128 : 256;
  if (train && T > Ts) {
    p.n_sub = 2;
    while (2 * (Ts - 16) + (p.n_sub - 2) * (Ts - 32) < T) ++p.n_sub;
  }
  p.B = B * p.n_sub;
  p.T = p.n_sub > 1 ? Ts : T;
  if (p.T <= 64) { p.nhalf = 2; p.MB = 64; p.NT = 1; }
  else { p.nhalf = 1; p.NT = (p.T > 128) ? 2 : 1; p.MB = 128 * p.NT; }
  p.HR = p.MB + 8;
  p.gh = (p.MB + 2) / (p.T + 2);
  const int wpt = p.nhalf * p.gh;
  p.n_tiles = (p.B + wpt - 1) / wpt;
  p.smem = (size_t)tile_smem_layout(g, p.nhalf * p.HR, train, split).total;
  p.ok = p.smem <= (size_t)225 * 1024;
  int per_sm = train ? 1 : (int)((size_t)220 * 1024 / (p.smem + 2048));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  p.grid = num_sms() * per_sm;
  if (p.grid > p.n_tiles) p.grid = p.n_tiles;
  return p;
}

static long long* g_dbg_timing = nullptr;
void set_debug_timing(long long* p) { g_dbg_timing = p; }

// Forward (plan.train false) and training: in the forward, the fields only training sets stay zero in `a`, and the
// sub-window fields (n_sub = 1, T_orig = T) select whole windows exactly as zero would.
int launch_tc_tile(const ConvArgs& a, const TilePlan& plan, cudaStream_t stream) {
  TcTileArgs p{};
  p.x = a.x; p.x_dtype = a.x_dtype; p.target = a.target; p.conf = a.conf; p.d_y = a.d_y; p.lengths = a.lengths;
  p.params = a.params; p.packed = a.packed; p.y = a.y; p.partials = a.partials; p.loss_partials = a.loss_partials;
  p.step_dev = a.step_dev; p.epoch_dev = a.epoch_dev; p.dbg = g_dbg_timing; p.fuse = a.fuse;
  p.win_start = a.wv.win_start; p.win_end = a.wv.win_end; p.n_frames = a.wv.n_frames; p.pad_mode = a.wv.pad_mode;
  p.T_orig = a.T; p.n_sub = plan.n_sub; p.loss_B = a.B;
  p.loss_kind = a.loss_kind; p.apply_mask = a.apply_mask; p.mode = a.mode; p.out_scale = a.out_scale; p.geo = a.geo;
  p.B = plan.B; p.T = plan.T;
  p.nhalf = plan.nhalf; p.MB = plan.MB; p.NT = plan.NT; p.HR = plan.HR; p.gh = plan.gh; p.n_tiles = plan.n_tiles;
  p.utt = a.utt; p.utt_seg = a.utt_seg; p.utt_max_len = a.utt_max_len;
  const bool train = plan.train, split = plan.split;
  const size_t smem = plan.smem;
  const int grid = plan.grid;
  // twenty-three instantiations: {forward, train, train over window views, forward over utterances} x {NT = 1, 2} x {bf16
  // operands, bf16 high/low pairs (fp32 mode)}, and training over segments with bf16 operands at NT = 1, 2 and with bf16
  // high/low pairs at NT = 1 (split training holds 128 rows, utterance_plan offers it no longer sub-window), and validation
  // over segments (a forward over utterances with loss_partials set) at NT = 1, 2 with both operand kinds
  const int nt2 = p.NT == 2 ? 1 : 0;
  const bool crit = !train && p.utt && p.loss_partials;
  const int kind = !train ? (p.utt ? (crit ? 5 : 3) : 0) : p.utt ? 4 : p.win_start ? 2 : 1;
  if (crit && p.gh != 1) { set_error("tile kernel: validation needs one sub-window per row segment (gh = %d)", p.gh); return B2H_ESHAPE; }
  const void* fns[6][2][2] = {
      {{(const void*)conv_tc_tile_kernel<false, 1, false>, (const void*)conv_tc_tile_kernel<false, 1, true>},
       {(const void*)conv_tc_tile_kernel<false, 2, false>, (const void*)conv_tc_tile_kernel<false, 2, true>}},
      {{(const void*)conv_tc_tile_kernel<true, 1, false>, (const void*)conv_tc_tile_kernel<true, 1, true>},
       {(const void*)conv_tc_tile_kernel<true, 2, false>, (const void*)conv_tc_tile_kernel<true, 2, true>}},
      {{(const void*)conv_tc_tile_kernel<true, 1, false, true>, (const void*)conv_tc_tile_kernel<true, 1, true, true>},
       {(const void*)conv_tc_tile_kernel<true, 2, false, true>, (const void*)conv_tc_tile_kernel<true, 2, true, true>}},
      {{(const void*)conv_tc_tile_kernel<false, 1, false, false, true>, (const void*)conv_tc_tile_kernel<false, 1, true, false, true>},
       {(const void*)conv_tc_tile_kernel<false, 2, false, false, true>, (const void*)conv_tc_tile_kernel<false, 2, true, false, true>}},
      {{(const void*)conv_tc_tile_kernel<true, 1, false, false, true>, (const void*)conv_tc_tile_kernel<true, 1, true, false, true>},
       {(const void*)conv_tc_tile_kernel<true, 2, false, false, true>, nullptr}},
      {{(const void*)conv_tc_tile_kernel<false, 1, false, false, true, true>, (const void*)conv_tc_tile_kernel<false, 1, true, false, true, true>},
       {(const void*)conv_tc_tile_kernel<false, 2, false, false, true, true>, (const void*)conv_tc_tile_kernel<false, 2, true, false, true, true>}}};
  const void* fn = fns[kind][nt2][split ? 1 : 0];
  if (!fn) { set_error("tile kernel: no instantiation for this plan"); return B2H_ESHAPE; }
  if (int rc = ensure_dyn_smem(fn, smem)) return rc;
  void* kargs[] = {&p};
  cudaError_t le;
  // The fused train step has a grid barrier inside: a cooperative launch guarantees that all its CTAs (<= 1 per SM)
  // are co-resident, also when other kernels share the device.
  // Forward launches are programmatic dependent launches: the kernel may start while its predecessor on the stream is
  // still running; it allocates TMEM, initialises its barriers and zeroes its shared memory, then blocks in
  // griddepcontrol.wait until the predecessor has completed (conv_tc_tile_kernel, part 1 / part 2).  Measured on B200
  // (profiles/r2_pdl.txt): forward B=512x64 10.7 -> 9.2 us per batch, B=1 latency 8.7 -> 7.3 us.  Train steps are
  // normal launches: PDL gained them only 0.3 us of 27.4 (their 128 CTAs hold one SM each, so only 20 of the next
  // step's CTAs find a free SM early, and the wait releases no sooner than a normal launch would start).
  const bool coop = train && p.fuse.enabled;
  const bool pdl = !train;
  if (pdl) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kTileThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    le = cudaLaunchKernelExC(&cfg, fn, kargs);
  } else if (coop) {
    le = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kTileThreads), kargs, smem, stream);
  } else {
    le = cudaLaunchKernel(fn, dim3(grid), dim3(kTileThreads), kargs, smem, stream);
  }
  if (le != cudaSuccess) { cudaGetLastError(); set_error("tile kernel launch: %s", cudaGetErrorString(le)); return B2H_ECUDA; }
  count_launch();
  return check_launch(train ? "conv_tc_tile_kernel<train>" : "conv_tc_tile_kernel<fwd>");
}

}  // namespace b2h
