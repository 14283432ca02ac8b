// extern "C" surface of libb2h.so (see include/b2h.h).  Argument checking, error reporting and
// dispatch between the fp32 (FFMA) and bf16 (tcgen05) kernels.  No CPU fallback exists anywhere.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <cmath>

#include "b2h_common.cuh"

namespace b2h {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return B2H_ECUDA;
  }
  return B2H_OK;
}
void count_launch(int n) { g_launches.fetch_add(n); }

// who == nullptr: a query, which leaves the error string alone
static bool geo_ok(int n_in, int C, int pos_emb, const char* who = nullptr) {
  if (n_in >= 1 && n_in <= 64 && C >= 1 && C <= B2H_MAX_C && pos_emb >= 0 && pos_emb <= 65536) return true;
  if (who) set_error("%s: unsupported geometry n_in=%d C=%d pos_emb=%d", who, n_in, C, pos_emb);
  return false;
}

// precision -> is it a tensor-core mode, and with bf16 high/low operand pairs (fp32 mode) or plain bf16 operands
static bool is_split(int precision) { return precision == B2H_FP32; }
static bool prec_ok(int precision) { return precision == B2H_FP32 || precision == B2H_BF16 || precision == B2H_FP32_FFMA; }

// Which kernel b2h_conv_forward launches and how (the ONE place that decides; b2h_kernel_choice reports it).
struct ForwardPlan {
  int kernel;
  TilePlan tile; RowspacePlan rowspace; WidePlan wide; FfmaPlan ffma;
};
static ForwardPlan forward_plan(const Geo& g, int B, int T, int precision) {
  ForwardPlan f{};
  f.tile = plan_tile(g, B, T, false, is_split(precision));   // independent 64/128/256-row tiles (T <= 256)
  f.rowspace = plan_rowspace(g, B, T);                         // long windows (T <= 1024): layer-major row space
  f.wide = plan_wide(g, B, T);                                 // wide models (C <= 256, T <= 256): streamed weights
  f.ffma = plan_ffma(g, B, T, false);
  f.kernel = B2H_KERNEL_NONE;
  if (precision == B2H_FP32_FFMA) {
    if (f.ffma.ok) f.kernel = B2H_KERNEL_FFMA;
  } else if (precision == B2H_FP32) {
    f.kernel = f.tile.ok ? B2H_KERNEL_TC_TILE : f.ffma.ok ? B2H_KERNEL_FFMA : B2H_KERNEL_NONE;
  } else if (precision == B2H_BF16) {
    f.kernel = f.tile.ok ? B2H_KERNEL_TC_TILE : f.rowspace.ok ? B2H_KERNEL_TC_ROWSPACE : f.wide.ok ? B2H_KERNEL_TC_WIDE : B2H_KERNEL_NONE;
  }
  return f;
}

// Which training path serves (B, T, C, precision) and how its workspace is laid out: the ONE place that decides.
//   [header B2H_WS_HEADER][gradient partials: nparts x gp_total floats][loss partials: n_loss floats][scratch (wide path)]
struct TrainPlan {
  int kernel;            // B2H_KERNEL_TC_TILE | B2H_KERNEL_TC_WIDE_TRAIN | B2H_KERNEL_FFMA | B2H_KERNEL_NONE
  TilePlan tile; WidePlan wide; FfmaPlan ffma;
  int nparts, n_loss;
  int64_t scratch_off, total;
};
static TrainPlan train_plan(const Geo& g, int B, int T, int precision) {
  TrainPlan t{};
  t.kernel = B2H_KERNEL_NONE;
  int64_t scratch = 0;
  if (precision == B2H_BF16 || precision == B2H_FP32) t.tile = plan_tile(g, B, T, true, is_split(precision));
  if (precision == B2H_BF16) t.wide = plan_wide(g, B, T);   // 32 < conv_channels <= 256: forward+criterion / dgrad chain / split-K wgrad
  t.ffma = plan_ffma(g, B, T, true);
  if (t.tile.ok) {
    t.kernel = B2H_KERNEL_TC_TILE; t.nparts = t.tile.grid; t.n_loss = t.nparts;
  } else if (t.wide.ok) {
    t.kernel = B2H_KERNEL_TC_WIDE_TRAIN; t.nparts = t.wide.ksplit; t.n_loss = t.wide.n_loss;
    scratch = t.wide.scratch_bytes;
  } else if (t.ffma.ok) {
    t.kernel = B2H_KERNEL_FFMA; t.nparts = t.ffma.grid; t.n_loss = t.nparts;
  }
  int64_t o = B2H_WS_HEADER + ((int64_t)t.nparts * gp_total(g) + t.n_loss) * 4;
  o = (o + 255) / 256 * 256;
  t.scratch_off = o;
  t.total = o + scratch + 256;
  return t;
}

// Which kernel and sub-window length b2h_conv_forward_utterances runs for n_utt utterances in a stream of n_frames frames:
// the ONE place that decides.  Per length Ts of the menu the family is the tile forward where it fits (bf16 and fp32 mode),
// else the wide forward (bf16 mode); the plan takes the Ts whose family computes the fewest MMA rows for an utterance of the
// mean length n_frames / n_utt under the cut rule (ties: the longer Ts, fewer sub-windows).  Rows per sub-window are the
// tile's rows over the windows it holds: 64 / 128 / 256 in the tile kernel, 256 / floor(258 / (Ts + 2)) in the wide one.
// Training over segments (kUttTrain, b2h_train_*_utterances): n_utt segments of at most max_len frames, the same rule for a
// segment of max_len frames over the lengths the tile kernel trains as whole windows (bf16: 64 / 128 / 256, fp32 mode: 64 /
// 128), sized for n_utt * n(max_len) sub-windows.  Validation over segments (kUttValidate, b2h_validate_utterances): the
// forward's families, the training's sizing.  The workspace layout is UttPlan's.
enum UttPurpose { kUttForward, kUttTrain, kUttValidate };
static UttPlan utterance_plan(const Geo& g, int64_t n_frames, int n_utt, int precision, UttPurpose purpose, int max_len) {
  static const int kMenu[3] = {256, 128, 64};
  UttPlan best{};
  best.kernel = B2H_KERNEL_NONE;
  if (precision != B2H_BF16 && precision != B2H_FP32) return best;   // the FFMA kernel reads dense windows only
  const bool train = purpose == kUttTrain, segments = purpose != kUttForward;
  if (segments && max_len < 1) return best;
  const int64_t mean = segments ? max_len : n_frames / (n_utt > 0 ? n_utt : 1);
  double best_rows = 0.0;
  for (int Ts : kMenu) {
    const int64_t max_sub = segments ? (int64_t)n_utt * sub_window_count(max_len, Ts)
                                     : (int64_t)(n_utt > 0 ? n_utt : 0) + n_frames / (Ts - 32);
    if (max_sub > (int64_t)INT32_MAX / 2) continue;
    UttPlan c{};
    c.Ts = Ts;
    c.max_sub = (int)max_sub;
    const int B = c.max_sub > 0 ? c.max_sub : 1;
    c.tile = plan_tile(g, B, Ts, train, is_split(precision));
    double rows_per_sub = 0.0;
    if (c.tile.ok && c.tile.n_sub == 1) {
      c.kernel = B2H_KERNEL_TC_TILE;
      rows_per_sub = (double)c.tile.MB / c.tile.gh;
    } else if (train) {
      continue;
    } else if (precision == B2H_BF16 && (c.wide = plan_wide(g, B, Ts)).ok) {
      c.kernel = B2H_KERNEL_TC_WIDE;
      rows_per_sub = 256.0 / c.wide.gh;
    } else {
      continue;
    }
    const double rows = rows_per_sub * sub_window_count(mean > 0 ? mean : 1, Ts);
    if (best.kernel != B2H_KERNEL_NONE && rows >= best_rows) continue;
    if (train) c.plan_off = (B2H_WS_HEADER + ((int64_t)c.tile.grid * gp_total(g) + c.tile.grid) * 4 + 255) / 256 * 256;
    c.seg_off = (utt_prefix_offset(c.max_sub) + 4 * ((int64_t)n_utt + 1) + 15) / 16 * 16;
    c.part_off = c.seg_off + (segments ? 8 * (int64_t)c.max_sub : 0);
    const int64_t end = c.part_off + (purpose == kUttValidate ? 4 * (int64_t)c.max_sub : 0);
    c.ws_bytes = (c.plan_off + end + 255) / 256 * 256;
    best = c;
    best_rows = rows;
  }
  return best;
}

// What utterance_plan serves, by purpose (the refusals of the queries and of the run entry points).
static const char* const kUttServed[3] = {
    "utterances are served in bf16 mode for conv_channels <= 256 and in fp32 mode for conv_channels <= 32 with at most 32 "
    "input channels",
    "segments are trained by the tile kernel: conv_channels <= 32 with at most 32 input channels, in bf16 or fp32 mode "
    "(wider models and fp32-ffma have no segment path)",
    "segments are validated by the utterance forward: in bf16 mode for conv_channels <= 256, in fp32 mode for "
    "conv_channels <= 32 with at most 32 input channels (fp32-ffma has no segment path)"};

// The six utterance queries: n utterances in a stream of n_frames frames (forward), or n segments of at most max_len frames.
// who == nullptr: a *_plan query, which leaves the error string alone, returns the kernel and writes the sub-window length
// to seg_len; else a *_workspace_bytes query, which returns the workspace size or B2H_ESHAPE.
static int64_t utterance_query(UttPurpose purpose, int64_t n_frames, int n, int max_len, int n_in, int C, int pos_emb,
                               int precision, int* seg_len, const char* who) {
  const int64_t refused = who ? B2H_ESHAPE : B2H_KERNEL_NONE;
  if (seg_len) *seg_len = 0;
  if (!geo_ok(n_in, C, pos_emb, who)) return refused;
  if (purpose == kUttForward ? n_frames < 0 || n_frames > INT32_MAX || n < 0 : n < 1 || max_len < 1) {
    if (who && purpose == kUttForward) set_error("%s: bad n_frames=%lld n_utt=%d", who, (long long)n_frames, n);
    else if (who) set_error("%s: bad n_seg=%d max_len=%d", who, n, max_len);
    return refused;
  }
  if (who && n == 0) return 256;     // the forward over no utterances launches nothing
  const UttPlan u = utterance_plan(make_geo(n_in, C, pos_emb), n_frames, n, precision, purpose, max_len);
  if (!who) {
    if (seg_len && u.kernel != B2H_KERNEL_NONE) *seg_len = u.Ts;
    return u.kernel;
  }
  if (u.kernel == B2H_KERNEL_NONE) {
    set_error("%s: %s (C=%d, n_in=%d, precision=%d)", who, kUttServed[purpose], C, n_in, precision);
    return B2H_ESHAPE;
  }
  return u.ws_bytes;
}

// The plan of an utterance run entry point over the sequences of sv: served, and the workspace large enough.
static int utterance_run_plan(const Geo& g, const SegmentView& sv, int precision, UttPurpose purpose, int64_t workspace_bytes,
                              const char* who, UttPlan* u) {
  *u = utterance_plan(g, sv.n_frames, sv.n, precision, purpose, sv.max_len);
  if (u->kernel == B2H_KERNEL_NONE) {
    set_error("%s: %s; no kernel for C=%d, n_in=%d, precision=%d", who, kUttServed[purpose], g.C, g.n_in, precision);
    return B2H_ESHAPE;
  }
  if (workspace_bytes < u->ws_bytes) {
    set_error("%s: workspace %lld B < %lld B", who, (long long)workspace_bytes, (long long)u->ws_bytes);
    return B2H_EWORKSPACE;
  }
  return B2H_OK;
}

}  // namespace b2h

using namespace b2h;

extern "C" const char* b2h_last_error(void) { return g_err; }
extern "C" int b2h_version(void) { return 100; }
extern "C" int64_t b2h_launch_count(void) { return g_launches.load(); }

extern "C" int b2h_device_ok(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) { cudaGetLastError(); return 0; }
  return major == 10 ? 1 : 0;
}

extern "C" int64_t b2h_param_count(int n_in, int C, int pos_emb) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_param_count")) return B2H_ESHAPE;
  return make_geo(n_in, C, pos_emb).P;
}
extern "C" int64_t b2h_param_offset(int n_in, int C, int pos_emb, int layer, int is_bias) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_param_offset")) return B2H_ESHAPE;
  if (layer < 1 || layer > 4) { set_error("b2h_param_offset: layer %d", layer); return B2H_EINVAL; }
  Geo g = make_geo(n_in, C, pos_emb);
  return is_bias ? g.b_off[layer - 1] : g.w_off[layer - 1];
}
/* Host-side self-check of the gradient-partial slot layout every training kernel writes (no GPU): every flat parameter
 * index maps to a distinct slot and back, every other slot decodes as padding.  gp_index_of_flat goes through
 * gp_slot_of_flat, the decode the packed-weight scatter uses, and gp_slot_in_layer, the slot the FFMA kernel writes.
 * Returns the number of violations (0 = consistent). */
extern "C" int64_t b2h_gp_layout_check(int n_in, int C, int pos_emb) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_gp_layout_check")) return B2H_ESHAPE;
  Geo g = make_geo(n_in, C, pos_emb);
  const int nj = gp_total(g);
  int64_t bad = (nj & 3) ? 1 : 0;
  for (int l = 0; l < 4; ++l) bad += (gp_layer_off(g, l) & 3) ? 1 : 0;
  int64_t real = 0;
  for (int j = 0; j < nj; ++j) {
    const int i = flat_index_of_gp(g, j);
    if (i < 0) continue;
    ++real;
    if (i >= g.P || gp_index_of_flat(g, i) != j) ++bad;
  }
  if (real != g.P) ++bad;
  for (int i = 0; i < g.P; ++i) {
    const int j = gp_index_of_flat(g, i);
    if (j < 0 || j >= nj || flat_index_of_gp(g, j) != i) ++bad;
  }
  return bad;
}
extern "C" int64_t b2h_packed_bytes(int n_in, int C, int pos_emb) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_packed_bytes")) return B2H_ESHAPE;
  return make_geo(n_in, C, pos_emb).packed_bytes;
}
extern "C" int b2h_supported(int T, int n_in, int C, int pos_emb, int precision) {
  if (!geo_ok(n_in, C, pos_emb) || T < 1 || !prec_ok(precision)) return 0;
  Geo g = make_geo(n_in, C, pos_emb);
  return (forward_plan(g, 1, T, precision).kernel != B2H_KERNEL_NONE && train_plan(g, 1, T, precision).kernel != B2H_KERNEL_NONE) ? 1 : 0;
}
extern "C" int b2h_forward_supported(int T, int n_in, int C, int pos_emb, int precision) {
  if (!geo_ok(n_in, C, pos_emb) || T < 1) return 0;
  return forward_plan(make_geo(n_in, C, pos_emb), 1, T, precision).kernel != B2H_KERNEL_NONE ? 1 : 0;
}
extern "C" int b2h_kernel_choice(int T, int n_in, int C, int pos_emb, int precision, int train) {
  if (!geo_ok(n_in, C, pos_emb) || T < 1) return B2H_KERNEL_NONE;
  Geo g = make_geo(n_in, C, pos_emb);
  if (!train) return forward_plan(g, 1, T, precision).kernel;
  if (!prec_ok(precision)) return B2H_KERNEL_NONE;
  return train_plan(g, 1, T, precision).kernel;
}
/* How the tile kernel's training path cuts a window of T frames (host-only query): returns n_sub (1 = whole windows) and,
 * for sub-window i, writes {first frame, first core row, end of the core rows (sub-window coordinates), sub-window length}. */
extern "C" int b2h_train_subwindows(int T, int n_in, int C, int pos_emb, int precision, int i, int* out4) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_train_subwindows")) return B2H_ESHAPE;
  if (T < 1) { set_error("b2h_train_subwindows: bad T"); return B2H_ESHAPE; }
  const TrainPlan t = train_plan(make_geo(n_in, C, pos_emb), 1, T, precision);
  const bool tile = t.kernel == B2H_KERNEL_TC_TILE;
  const int n = tile ? t.tile.n_sub : 1, Ts = tile ? t.tile.T : T;
  if (out4) {
    if (i < 0 || i >= n) { set_error("b2h_train_subwindows: sub-window %d of %d", i, n); return B2H_EINVAL; }
    const SubWindow s = sub_window(T, Ts, n, i);
    out4[0] = s.start; out4[1] = s.clo; out4[2] = s.chi; out4[3] = Ts;
  }
  return n;
}

extern "C" int64_t b2h_workspace_bytes(int B, int T, int n_in, int C, int pos_emb, int precision) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_workspace_bytes")) return B2H_ESHAPE;
  if (B < 1 || T < 1) return B2H_WS_HEADER + 256;
  return train_plan(make_geo(n_in, C, pos_emb), B, T, precision).total;
}

extern "C" int b2h_pack_weights(const float* params, void* packed, int n_in, int C, int pos_emb, void* stream) {
  if (!params || !packed) { set_error("b2h_pack_weights: null pointer"); return B2H_EINVAL; }
  if (!geo_ok(n_in, C, pos_emb, "b2h_pack_weights")) return B2H_ESHAPE;
  return launch_pack(params, packed, make_geo(n_in, C, pos_emb), (cudaStream_t)stream);
}

// The window view of the *_windows entry points.
static WindowView window_view(const int64_t* win_start, const int64_t* win_end, int64_t n_frames, int pad_mode) {
  return WindowView{reinterpret_cast<const long long*>(win_start), reinterpret_cast<const long long*>(win_end), (long long)n_frames, pad_mode};
}

// The segment view of the *_utterances entry points (the forward's offsets: seg_end = offsets + 1, max_len = 0).
static SegmentView segment_view(const int64_t* seg_start, const int64_t* seg_end, int n, int64_t n_frames, int max_len) {
  return SegmentView{reinterpret_cast<const long long*>(seg_start), reinterpret_cast<const long long*>(seg_end), n, (long long)n_frames, max_len};
}

// The checks every forward and training entry point makes first, in this order: pointers (`out` = y in the forward, the
// workspace in training), x_dtype, pad_mode, geometry, shape (B >= B_min; a segment view: n >= B_min sequences in a stream
// of at most INT32_MAX frames, and with B_min = 1, segments of max_len >= 1 frames).
static int check_common(const void* x, int x_dtype, const WindowView* wv, const SegmentView* sv, const float* params,
                        const void* packed, const void* out, int B, int B_min, int T, int n_in, int C, int pos_emb,
                        const char* who) {
  if (!x || (wv && !wv->win_start) || (sv && (!sv->seg_a || !sv->seg_b)) || !params || !packed || !out) {
    set_error("%s: null pointer", who);
    return B2H_EINVAL;
  }
  if (x_dtype != B2H_DT_F32 && x_dtype != B2H_DT_BF16) { set_error("%s: bad x_dtype %d", who, x_dtype); return B2H_EINVAL; }
  if (wv && wv->pad_mode != B2H_PAD_REPEAT_FIRST && wv->pad_mode != B2H_PAD_ZEROS) { set_error("%s: bad pad_mode %d", who, wv->pad_mode); return B2H_EINVAL; }
  if (!geo_ok(n_in, C, pos_emb, who)) return B2H_ESHAPE;
  if (sv) {
    if (sv->n < B_min || sv->n_frames < 0 || sv->n_frames > INT32_MAX || (B_min > 0 && sv->max_len < 1)) {
      if (B_min > 0) set_error("%s: bad n_seg=%d max_len=%d n_frames=%lld", who, sv->n, sv->max_len, sv->n_frames);
      else set_error("%s: bad n_utt=%d n_frames=%lld", who, sv->n, sv->n_frames);
      return B2H_ESHAPE;
    }
  } else if (B < B_min || T < 1 || (wv && wv->n_frames < 0)) {
    set_error("%s: bad B=%d T=%d", who, B, T);
    return B2H_ESHAPE;
  }
  return B2H_OK;
}

static bool misaligned(const void* p, uintptr_t mask) { return reinterpret_cast<uintptr_t>(p) & mask; }

// The forward of B dense windows x (wv == nullptr), of B windows viewed in the frame stream x, or of the B = sv->n
// utterances of a segment view (T unused; the plan's table lives in the workspace).  Views are read by the tensor-core
// kernels only: fp32 mode beyond the tile kernel runs on FFMA, which reads dense windows.
static int conv_forward(const void* x, int x_dtype, const WindowView* wv, const SegmentView* sv, const float* params,
                        const void* packed, const int32_t* lengths, float* y, int B, int T, int n_in, int C, int pos_emb,
                        int precision, int apply_mask, float out_scale, void* workspace, int64_t workspace_bytes,
                        cudaStream_t stream, const char* who) {
  if (int rc = check_common(x, x_dtype, wv, sv, params, packed, y, B, 0, T, n_in, C, pos_emb, who)) return rc;
  if (apply_mask && !lengths) { set_error("%s: apply_mask needs lengths", who); return B2H_EINVAL; }
  if (B == 0) return B2H_OK;
  if (misaligned(x, 15) || misaligned(y, 15) || misaligned(packed, 15) || (sv && (misaligned(workspace, 15) || misaligned(sv->seg_a, 7)))) {
    if (sv) set_error("%s: frames, y, packed and workspace must be 16-byte aligned, offsets 8-byte aligned", who);
    else set_error("%s: %s, y and packed must be 16-byte aligned", who, wv ? "frames" : "x");
    return B2H_EALIGN;
  }
  if (!prec_ok(precision)) { set_error("%s: bad precision %d", who, precision); return B2H_EINVAL; }
  ConvArgs a{};
  a.x = x; a.x_dtype = x_dtype; a.lengths = lengths; a.params = params; a.packed = reinterpret_cast<const char*>(packed);
  a.y = y; a.B = B; a.T = T; a.apply_mask = apply_mask; a.mode = 0; a.out_scale = out_scale;
  a.geo = make_geo(n_in, C, pos_emb);
  if (wv) a.wv = *wv;
  if (sv) {
    UttPlan u;
    if (int rc = utterance_run_plan(a.geo, *sv, precision, kUttForward, workspace_bytes, who, &u)) return rc;
    return launch_utterances(a, u, *sv, workspace, nullptr, nullptr, stream);
  }
  const ForwardPlan f = forward_plan(a.geo, B, T, precision);
  if (f.kernel == B2H_KERNEL_TC_TILE) return launch_tc_tile(a, f.tile, stream);
  if (f.kernel == B2H_KERNEL_TC_WIDE) return launch_tc_wide_fwd(a, f.wide, stream);
  if (f.kernel == B2H_KERNEL_TC_ROWSPACE) return launch_tc_fwd(a, f.rowspace, stream);
  if (f.kernel == B2H_KERNEL_FFMA && !wv) return launch_fp32(a, f.ffma, stream);
  if (wv)
    set_error("%s: window views are served in bf16 mode for conv_channels <= 256 with T <= 256, <= 48 with T <= 640 and <= 32 "
              "with T <= 1024 (the last two with at most 32 input channels), in fp32 mode for conv_channels <= 32 with T <= 256; "
              "materialise the windows (b2h_preprocess) for C=%d, T=%d, precision=%d", who, C, T, precision);
  else
    set_error("%s: no kernel for C=%d, T=%d, precision=%d (tensor cores: bf16 conv_channels <= 256 with T <= 256, <= 48 with "
              "T <= 640 and <= 32 with T <= 1024 at up to 32 input channels, fp32 conv_channels <= 32 with T <= 256; the FFMA "
              "kernel would need %zu B of its 226 KB of shared memory)", who, C, T, precision, f.ffma.smem);
  return B2H_ESHAPE;
}

extern "C" int b2h_conv_forward(const void* x, int x_dtype, const float* params, const void* packed, const int32_t* lengths,
                                float* y, int B, int T, int n_in, int C, int pos_emb, int precision, int apply_mask,
                                float out_scale, void* stream) {
  return conv_forward(x, x_dtype, nullptr, nullptr, params, packed, lengths, y, B, T, n_in, C, pos_emb, precision, apply_mask,
                      out_scale, nullptr, 0, (cudaStream_t)stream, "b2h_conv_forward");
}

extern "C" int b2h_conv_forward_windows(const void* frames, int x_dtype, int64_t n_frames, const int64_t* win_start,
                                        const int64_t* win_end, int pad_mode, const float* params, const void* packed,
                                        const int32_t* lengths, float* y, int n_win, int T, int n_in, int C, int pos_emb,
                                        int precision, int apply_mask, float out_scale, void* stream) {
  const WindowView wv = window_view(win_start, win_end, n_frames, pad_mode);
  return conv_forward(frames, x_dtype, &wv, nullptr, params, packed, lengths, y, n_win, T, n_in, C, pos_emb, precision,
                      apply_mask, out_scale, nullptr, 0, (cudaStream_t)stream, "b2h_conv_forward_windows");
}

extern "C" int b2h_utterances_plan(int64_t n_frames, int n_utt, int n_in, int C, int pos_emb, int precision, int* seg_len) {
  return (int)utterance_query(kUttForward, n_frames, n_utt, 0, n_in, C, pos_emb, precision, seg_len, nullptr);
}

extern "C" int b2h_utterance_subwindows(int L, int Ts, int i, int* out3) {
  if (L < 0 || Ts <= 32) { set_error("b2h_utterance_subwindows: bad L=%d Ts=%d", L, Ts); return B2H_ESHAPE; }
  const int n = sub_window_count(L, Ts);
  if (out3) {
    if (i < 0 || i >= n) { set_error("b2h_utterance_subwindows: sub-window %d of %d", i, n); return B2H_EINVAL; }
    if (n == 1) { out3[0] = 0; out3[1] = 0; out3[2] = L; }
    else {
      const SubWindow s = sub_window(L, Ts, n, i);
      out3[0] = s.start; out3[1] = s.clo; out3[2] = s.chi;
    }
  }
  return n;
}

extern "C" int64_t b2h_utterances_workspace_bytes(int64_t n_frames, int n_utt, int n_in, int C, int pos_emb, int precision) {
  return utterance_query(kUttForward, n_frames, n_utt, 0, n_in, C, pos_emb, precision, nullptr, "b2h_utterances_workspace_bytes");
}

extern "C" int b2h_conv_forward_utterances(const void* frames, int x_dtype, int64_t n_frames, const int64_t* offsets, int n_utt,
                                           const float* params, const void* packed, float* y, int n_in, int C, int pos_emb,
                                           int precision, float out_scale, void* workspace, int64_t workspace_bytes,
                                           void* stream) {
  const char* who = "b2h_conv_forward_utterances";
  if (!workspace) { set_error("%s: null pointer", who); return B2H_EINVAL; }
  const SegmentView sv = segment_view(offsets, offsets ? offsets + 1 : nullptr, n_utt, n_frames, 0);
  return conv_forward(frames, x_dtype, nullptr, &sv, params, packed, nullptr, y, n_utt, 0, n_in, C, pos_emb, precision, 0,
                      out_scale, workspace, workspace_bytes, (cudaStream_t)stream, who);
}

// What a training launch left for the reduction / Adam launches that follow it (rc != B2H_OK: nothing was launched).
struct TrainResult {
  int rc;
  Geo g;
  TrainPlan plan;
  float* partials;        // gradient partials in the workspace: plan.nparts slices of gp_total(g) floats
  float* loss_partials;   // plan.n_loss floats
};

// The criterion's inputs of training and validation: target rows, the windows' lengths (not for segments, which carry their
// own), loss_kind and, for confL1, the confidence rows.
static int check_criterion(const float* target, const float* conf, const int32_t* lengths, bool need_lengths, int loss_kind,
                           const char* who) {
  if (!target || (need_lengths && !lengths)) { set_error(need_lengths ? "%s: null target/lengths" : "%s: null target", who); return B2H_EINVAL; }
  if (loss_kind != B2H_LOSS_L1 && loss_kind != B2H_LOSS_CONFL1) { set_error("%s: bad loss_kind %d", who, loss_kind); return B2H_EINVAL; }
  if (loss_kind == B2H_LOSS_CONFL1 && !conf) { set_error("%s: confL1 needs scores", who); return B2H_EINVAL; }
  return B2H_OK;
}

// The training forward + criterion + backward of B dense windows (wv == nullptr), of B windows viewed in the frame streams
// x / target / conf, or of the segments of sv in them, each trained as one sequence (views: mode 1 only; the tensor-core
// kernels only: the FFMA kernel reads dense windows; segments: the tile kernel, the plan's table in the workspace past the
// partials).  fuse != nullptr asks the tile kernel to reduce and apply Adam in the same launch.
static TrainResult train_common(const void* x, int x_dtype, const WindowView* wv, const SegmentView* sv, const float* target,
                                const float* conf, const float* d_y, const int32_t* lengths, const float* params,
                                const void* packed, float* pred_out, int B, int T, int n_in, int C, int pos_emb, int loss_kind,
                                int precision, int mode, void* workspace, int64_t workspace_bytes, cudaStream_t stream,
                                const char* who, long long* step_dev, long long* epoch_dev, const FuseAdam* fuse) {
  TrainResult r{};
  auto result = [&r](int rc) { r.rc = rc; return r; };
  if (int rc = check_common(x, x_dtype, wv, sv, params, packed, workspace, B, 1, T, n_in, C, pos_emb, who)) return result(rc);
  if (!prec_ok(precision)) { set_error("%s: bad precision %d", who, precision); return result(B2H_EINVAL); }
  if (mode == 1) {
    if (int rc = check_criterion(target, conf, lengths, !sv, loss_kind, who)) return result(rc);
  } else if (!d_y) { set_error("%s: null d_y", who); return result(B2H_EINVAL); }
  // A stream's target row (168 B) and confidence row (84 B) start 8 / 4 bytes past a 16-B boundary at odd frames: the
  // kernels read them with float2 / float loads and use a bulk copy only where the address allows it.
  const bool stream_rows = wv || sv;
  if (misaligned(x, 15) || misaligned(target, stream_rows ? 7 : 15) || misaligned(conf, stream_rows ? 3 : 0) || misaligned(packed, 15) ||
      (sv && (misaligned(pred_out, 15) || misaligned(workspace, 15) || misaligned(sv->seg_a, 7) || misaligned(sv->seg_b, 7)))) {
    if (sv)
      set_error("%s: frames, packed, pred_out and workspace must be 16-byte aligned, target_frames, seg_start and seg_end 8-byte "
                "and conf_frames 4-byte aligned", who);
    else if (wv) set_error("%s: frames and packed must be 16-byte aligned, target_frames 8-byte and conf_frames 4-byte aligned", who);
    else set_error("%s: x, target and packed must be 16-byte aligned", who);
    return result(B2H_EALIGN);
  }
  r.g = make_geo(n_in, C, pos_emb);
  TrainPlan& plan = r.plan;
  UttPlan u{};
  if (sv) {
    if (int rc = utterance_run_plan(r.g, *sv, precision, kUttTrain, workspace_bytes, who, &u)) return result(rc);
    plan.kernel = B2H_KERNEL_TC_TILE; plan.tile = u.tile; plan.nparts = plan.n_loss = u.tile.grid;
  } else {
    plan = train_plan(r.g, B, T, precision);
    if (wv && plan.kernel != B2H_KERNEL_TC_TILE && plan.kernel != B2H_KERNEL_TC_WIDE_TRAIN) {
      set_error("%s: window views are trained on the tensor cores: in bf16 mode for conv_channels <= 32 with at most 32 input "
                "channels and T <= 4096, and for conv_channels <= 256 with T <= 256; in fp32 mode for conv_channels <= 32 with "
                "at most 32 input channels and T <= 4096; materialise the windows (b2h_preprocess) for C=%d, T=%d, precision=%d",
                who, C, T, precision);
      return result(B2H_ESHAPE);
    }
    if (plan.kernel == B2H_KERNEL_NONE) {
      set_error("%s: no training kernel for conv_channels=%d, T=%d, precision=%d (tcgen05 training: C <= 32 in the one-launch "
                "tile kernel, C <= 256 in bf16 mode through the wide kernels, T <= 256; the FFMA kernel would need %zu B of "
                "shared memory)", who, C, T, precision, plan.ffma.smem);
      return result(B2H_ESHAPE);
    }
    if (workspace_bytes < plan.total - 256) { set_error("%s: workspace %lld B < %lld B", who, (long long)workspace_bytes, (long long)plan.total); return result(B2H_EWORKSPACE); }
    if (misaligned(workspace, 15)) { set_error("%s: workspace must be 16-byte aligned", who); return result(B2H_EALIGN); }
  }
  // [header: launch sequence + per-CTA arrival flags of the fused kernel, FIXED offset][gradient partials][loss partials]
  // [scratch (wide) | the utterance plan's table (segments)]
  r.partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + B2H_WS_HEADER);
  r.loss_partials = r.partials + (size_t)plan.nparts * gp_total(r.g);
  if (sv && pred_out) {   // the masked prediction (n_seg, max_len, 42): rows at or past a segment's end stay zero
    const cudaError_t e = cudaMemsetAsync(pred_out, 0, (size_t)sv->n * sv->max_len * B2H_COUT * 4, stream);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("%s: cudaMemsetAsync: %s", who, cudaGetErrorString(e)); return result(B2H_ECUDA); }
  }
  ConvArgs a{};
  a.x = x; a.x_dtype = x_dtype; a.target = target; a.conf = conf; a.d_y = d_y; a.lengths = lengths; a.params = params;
  a.packed = reinterpret_cast<const char*>(packed); a.y = pred_out; a.partials = r.partials; a.loss_partials = r.loss_partials;
  a.B = B; a.T = T; a.loss_kind = loss_kind; a.apply_mask = 1; a.mode = mode; a.out_scale = 1.0f; a.geo = r.g;
  a.step_dev = step_dev;
  a.epoch_dev = epoch_dev;
  if (wv) a.wv = *wv;
  if (plan.kernel == B2H_KERNEL_TC_TILE) {
    if (fuse) {
      if (plan.nparts > B2H_WS_MAX_CTA) { set_error("%s: %d CTAs exceed the %d arrival flags of the workspace header", who, plan.nparts, B2H_WS_MAX_CTA); return result(B2H_ESHAPE); }
      a.fuse = *fuse;
      a.fuse.enabled = 1;
      a.fuse.hdr = reinterpret_cast<unsigned*>(workspace);
    }
    if (sv) {
      return result(launch_utterances(a, u, *sv, reinterpret_cast<char*>(workspace) + u.plan_off, nullptr, nullptr, stream));
    }
    return result(launch_tc_tile(a, plan.tile, stream));
  }
  if (plan.kernel == B2H_KERNEL_TC_WIDE_TRAIN) {
    // (the forward+criterion kernel's CTA 0 bumps the device-side step / epoch counters the Adam kernels read)
    return result(launch_tc_wide_train(a, plan.wide, reinterpret_cast<unsigned char*>(workspace) + plan.scratch_off, stream));
  }
  return result(launch_fp32(a, plan.ffma, stream));
}

static int train_forward_backward(const void* x, int x_dtype, const WindowView* wv, const SegmentView* sv, const float* target,
                                  const float* conf, const int32_t* lengths, const float* params, const void* packed,
                                  float* grads_out, float* loss_out, float* pred_out, int B, int T, int n_in, int C, int pos_emb,
                                  int loss_kind, int precision, int64_t* step_dev, void* workspace, int64_t workspace_bytes,
                                  void* stream, const char* who) {
  if (grads_out && !loss_out) { set_error("%s: null loss_out", who); return B2H_EINVAL; }
  const TrainResult r = train_common(x, x_dtype, wv, sv, target, conf, nullptr, lengths, params, packed, pred_out, B, T, n_in, C,
                                     pos_emb, loss_kind, precision, 1, workspace, workspace_bytes, (cudaStream_t)stream, who,
                                     reinterpret_cast<long long*>(step_dev), nullptr, nullptr);
  if (r.rc || !grads_out) return r.rc;   // grads_out == NULL: only the fused kernel runs, partials stay in the workspace
  return launch_reduce(r.partials, r.plan.nparts, r.g, grads_out, r.loss_partials, r.plan.n_loss, loss_out, nullptr,
                       (cudaStream_t)stream);
}

extern "C" int b2h_train_forward_backward(const void* x, int x_dtype, const float* target, const float* conf,
                                          const int32_t* lengths, const float* params, const void* packed,
                                          float* grads_out, float* loss_out, float* pred_out, int B, int T, int n_in,
                                          int C, int pos_emb, int loss_kind, int precision, int64_t* step_dev,
                                          void* workspace, int64_t workspace_bytes, void* stream) {
  return train_forward_backward(x, x_dtype, nullptr, nullptr, target, conf, lengths, params, packed, grads_out, loss_out,
                                pred_out, B, T, n_in, C, pos_emb, loss_kind, precision, step_dev, workspace, workspace_bytes,
                                stream, "b2h_train_forward_backward");
}

extern "C" int b2h_train_forward_backward_windows(const void* frames, int x_dtype, const float* target_frames,
                                                  const float* conf_frames, int64_t n_frames, const int64_t* win_start,
                                                  const int64_t* win_end, int pad_mode, const int32_t* lengths,
                                                  const float* params, const void* packed, float* grads_out, float* loss_out,
                                                  float* pred_out, int n_win, int T, int n_in, int C, int pos_emb,
                                                  int loss_kind, int precision, int64_t* step_dev, void* workspace,
                                                  int64_t workspace_bytes, void* stream) {
  const WindowView wv = window_view(win_start, win_end, n_frames, pad_mode);
  return train_forward_backward(frames, x_dtype, &wv, nullptr, target_frames, conf_frames, lengths, params, packed, grads_out,
                                loss_out, pred_out, n_win, T, n_in, C, pos_emb, loss_kind, precision, step_dev, workspace,
                                workspace_bytes, stream, "b2h_train_forward_backward_windows");
}

extern "C" int64_t b2h_dp_exchange_floats(int n_in, int C, int pos_emb, int world) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_dp_exchange_floats")) return B2H_ESHAPE;
  if (world < 1 || world > 32) { set_error("b2h_dp_exchange_floats: bad world"); return B2H_EINVAL; }
  Geo g = make_geo(n_in, C, pos_emb);
  // one-launch tile path: 4-byte words [2][world][slots] = 2*world*slots floats (the size returned is twice that); the
  // three-launch path needs [2][P] fp32 + [world] int64 flags, which is smaller
  return 4 * (int64_t)world * gp_total(g) + 64;
}

extern "C" int64_t b2h_dp_exchange_fill(int T, int n_in, int C, int pos_emb, int precision) {
  if (!geo_ok(n_in, C, pos_emb, "b2h_dp_exchange_fill")) return B2H_ESHAPE;
  // fused tile kernel: every 32-bit word starts as the "not arrived" sentinel; three-launch path: zeroed gradients + flags
  return train_plan(make_geo(n_in, C, pos_emb), 1, T, precision).kernel == B2H_KERNEL_TC_TILE ? 0xFFFFFFFFll : 0ll;
}

extern "C" int b2h_dp_status(void) { return dp_status_and_clear(); }

extern "C" int b2h_conv_backward(const void* x, int x_dtype, const float* d_y, const float* params, const void* packed,
                                 float* grads_out, int B, int T, int n_in, int C, int pos_emb, int precision,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  if (!grads_out) { set_error("b2h_conv_backward: null output"); return B2H_EINVAL; }
  const TrainResult r = train_common(x, x_dtype, nullptr, nullptr, nullptr, nullptr, d_y, nullptr, params, packed, nullptr, B, T,
                                     n_in, C, pos_emb, 0, precision, 2, workspace, workspace_bytes, (cudaStream_t)stream,
                                     "b2h_conv_backward", nullptr, nullptr, nullptr);
  if (r.rc) return r.rc;
  return launch_reduce(r.partials, r.plan.nparts, r.g, grads_out, nullptr, r.plan.n_loss, nullptr, nullptr, (cudaStream_t)stream);
}

// The Adam tail of the fused tile kernel (train_common enables it and points it at the workspace header).
static FuseAdam fuse_adam(float* params, void* packed, float* exp_avg, float* exp_avg_sq, float* loss_out, double lr,
                          double beta1, double beta2, double eps, float grad_scale, int64_t* step_dev, const double* lr_dev) {
  FuseAdam f{};
  f.params = params; f.m = exp_avg; f.v = exp_avg_sq; f.packed = reinterpret_cast<char*>(packed);
  f.lr = lr; f.beta1 = beta1; f.beta2 = beta2; f.eps = (float)eps; f.grad_scale = grad_scale;
  f.lr_dev = lr_dev;
  f.step_dev = reinterpret_cast<const long long*>(step_dev); f.loss_out = loss_out; f.world = 1;
  return f;
}

static int train_step(const void* x, int x_dtype, const WindowView* wv, const SegmentView* sv, const float* target,
                      const float* conf, const int32_t* lengths, float* params, void* packed, float* exp_avg, float* exp_avg_sq,
                      float* loss_out, int B, int T, int n_in, int C, int pos_emb, int loss_kind, int precision, double lr,
                      double beta1, double beta2, double eps, int64_t step, int64_t* step_dev, const double* lr_dev,
                      void* workspace, int64_t workspace_bytes, void* stream, const char* who) {
  if (!exp_avg || !exp_avg_sq || !loss_out) { set_error("%s: null pointer", who); return B2H_EINVAL; }
  if (step < 1 && !step_dev) { set_error("%s: step must be >= 1", who); return B2H_EINVAL; }
  // segments have the fused step only: it reads the Adam step from the device counter and advances it (a refused segment
  // list leaves it alone)
  if (sv && !step_dev) { set_error("%s: null step_dev (the fused step reads and advances the device-side step counter)", who); return B2H_EINVAL; }
  // tile kernel + device-side step counter: ONE cooperative launch (reduction + Adam + re-pack in its tail)
  const FuseAdam fuse = fuse_adam(params, packed, exp_avg, exp_avg_sq, loss_out, lr, beta1, beta2, eps, 1.0f, step_dev, lr_dev);
  const TrainResult r = train_common(x, x_dtype, wv, sv, target, conf, nullptr, lengths, params, packed, nullptr, B, T, n_in, C,
                                     pos_emb, loss_kind, precision, 1, workspace, workspace_bytes, (cudaStream_t)stream, who,
                                     reinterpret_cast<long long*>(step_dev), nullptr, step_dev ? &fuse : nullptr);
  if (r.rc) return r.rc;
  if (step_dev && r.plan.kernel == B2H_KERNEL_TC_TILE) return B2H_OK;
  return launch_adam_partials(params, r.partials, r.plan.nparts, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, step < 1 ? 1 : step,
                              reinterpret_cast<const long long*>(step_dev), lr_dev, packed, r.g, r.loss_partials, r.plan.n_loss,
                              loss_out, (cudaStream_t)stream);
}

extern "C" int b2h_train_step(const void* x, int x_dtype, const float* target, const float* conf, const int32_t* lengths,
                              float* params, void* packed, float* exp_avg, float* exp_avg_sq, float* loss_out, int B,
                              int T, int n_in, int C, int pos_emb, int loss_kind, int precision, double lr, double beta1,
                              double beta2, double eps, int64_t step, int64_t* step_dev, const double* lr_dev, void* workspace,
                              int64_t workspace_bytes, void* stream) {
  return train_step(x, x_dtype, nullptr, nullptr, target, conf, lengths, params, packed, exp_avg, exp_avg_sq, loss_out, B, T, n_in,
                    C, pos_emb, loss_kind, precision, lr, beta1, beta2, eps, step, step_dev, lr_dev, workspace, workspace_bytes,
                    stream, "b2h_train_step");
}

extern "C" int b2h_train_step_windows(const void* frames, int x_dtype, const float* target_frames, const float* conf_frames,
                                      int64_t n_frames, const int64_t* win_start, const int64_t* win_end, int pad_mode,
                                      const int32_t* lengths, float* params, void* packed, float* exp_avg, float* exp_avg_sq,
                                      float* loss_out, int n_win, int T, int n_in, int C, int pos_emb, int loss_kind,
                                      int precision, double lr, double beta1, double beta2, double eps, int64_t step,
                                      int64_t* step_dev, const double* lr_dev, void* workspace, int64_t workspace_bytes,
                                      void* stream) {
  const WindowView wv = window_view(win_start, win_end, n_frames, pad_mode);
  return train_step(frames, x_dtype, &wv, nullptr, target_frames, conf_frames, lengths, params, packed, exp_avg, exp_avg_sq,
                    loss_out, n_win, T, n_in, C, pos_emb, loss_kind, precision, lr, beta1, beta2, eps, step, step_dev, lr_dev,
                    workspace, workspace_bytes, stream, "b2h_train_step_windows");
}

extern "C" int b2h_train_utterances_plan(int n_seg, int max_len, int n_in, int C, int pos_emb, int precision, int* seg_len) {
  return (int)utterance_query(kUttTrain, 0, n_seg, max_len, n_in, C, pos_emb, precision, seg_len, nullptr);
}

extern "C" int64_t b2h_train_utterances_workspace_bytes(int n_seg, int max_len, int n_in, int C, int pos_emb, int precision) {
  return utterance_query(kUttTrain, 0, n_seg, max_len, n_in, C, pos_emb, precision, nullptr, "b2h_train_utterances_workspace_bytes");
}

extern "C" int b2h_train_forward_backward_utterances(const void* frames, int x_dtype, const float* target_frames,
                                                     const float* conf_frames, int64_t n_frames, const int64_t* seg_start,
                                                     const int64_t* seg_end, int n_seg, int max_len, const float* params,
                                                     const void* packed, float* grads_out, float* loss_out, float* pred_out,
                                                     int n_in, int C, int pos_emb, int loss_kind, int precision,
                                                     int64_t* step_dev, void* workspace, int64_t workspace_bytes, void* stream) {
  const char* who = "b2h_train_forward_backward_utterances";
  if (!grads_out || !loss_out) { set_error("%s: null pointer", who); return B2H_EINVAL; }
  const SegmentView sv = segment_view(seg_start, seg_end, n_seg, n_frames, max_len);
  return train_forward_backward(frames, x_dtype, nullptr, &sv, target_frames, conf_frames, nullptr, params, packed, grads_out,
                                loss_out, pred_out, n_seg, 1, n_in, C, pos_emb, loss_kind, precision, step_dev, workspace,
                                workspace_bytes, stream, who);
}

extern "C" int b2h_train_step_utterances(const void* frames, int x_dtype, const float* target_frames, const float* conf_frames,
                                         int64_t n_frames, const int64_t* seg_start, const int64_t* seg_end, int n_seg,
                                         int max_len, float* params, void* packed, float* exp_avg, float* exp_avg_sq,
                                         float* loss_out, int n_in, int C, int pos_emb, int loss_kind, int precision, double lr,
                                         double beta1, double beta2, double eps, int64_t step, int64_t* step_dev,
                                         const double* lr_dev, void* workspace, int64_t workspace_bytes, void* stream) {
  const SegmentView sv = segment_view(seg_start, seg_end, n_seg, n_frames, max_len);
  return train_step(frames, x_dtype, nullptr, &sv, target_frames, conf_frames, nullptr, params, packed, exp_avg, exp_avg_sq,
                    loss_out, n_seg, 1, n_in, C, pos_emb, loss_kind, precision, lr, beta1, beta2, eps, step, step_dev, lr_dev,
                    workspace, workspace_bytes, stream, "b2h_train_step_utterances");
}

extern "C" int b2h_validate_utterances_plan(int n_seg, int max_len, int n_in, int C, int pos_emb, int precision, int* seg_len) {
  return (int)utterance_query(kUttValidate, 0, n_seg, max_len, n_in, C, pos_emb, precision, seg_len, nullptr);
}

extern "C" int64_t b2h_validate_utterances_workspace_bytes(int n_seg, int max_len, int n_in, int C, int pos_emb, int precision) {
  return utterance_query(kUttValidate, 0, n_seg, max_len, n_in, C, pos_emb, precision, nullptr,
                         "b2h_validate_utterances_workspace_bytes");
}

// Validation over segments: the forward over them with the criterion per sub-window instead of predictions, then the
// per-segment means and the loss.
extern "C" int b2h_validate_utterances(const void* frames, int x_dtype, const float* target_frames, const float* conf_frames,
                                       int64_t n_frames, const int64_t* seg_start, const int64_t* seg_end, int n_seg, int max_len,
                                       const float* params, const void* packed, float* seg_loss_out, float* loss_out, int n_in,
                                       int C, int pos_emb, int loss_kind, int precision, void* workspace,
                                       int64_t workspace_bytes, void* stream) {
  const char* who = "b2h_validate_utterances";
  if (!loss_out) { set_error("%s: null pointer", who); return B2H_EINVAL; }
  const SegmentView sv = segment_view(seg_start, seg_end, n_seg, n_frames, max_len);
  if (int rc = check_common(frames, x_dtype, nullptr, &sv, params, packed, workspace, n_seg, 1, 1, n_in, C, pos_emb, who)) return rc;
  if (!prec_ok(precision)) { set_error("%s: bad precision %d", who, precision); return B2H_EINVAL; }
  if (int rc = check_criterion(target_frames, conf_frames, nullptr, false, loss_kind, who)) return rc;
  if (misaligned(frames, 15) || misaligned(target_frames, 7) || misaligned(conf_frames, 3) || misaligned(packed, 15) ||
      misaligned(workspace, 15) || misaligned(seg_start, 7) || misaligned(seg_end, 7) || misaligned(seg_loss_out, 3) ||
      misaligned(loss_out, 3)) {
    set_error("%s: frames, packed and workspace must be 16-byte aligned, target_frames, seg_start and seg_end 8-byte, "
              "conf_frames, seg_loss_out and loss_out 4-byte aligned", who);
    return B2H_EALIGN;
  }
  ConvArgs a{};
  a.x = frames; a.x_dtype = x_dtype; a.target = target_frames; a.conf = conf_frames; a.params = params;
  a.packed = reinterpret_cast<const char*>(packed); a.loss_kind = loss_kind; a.mode = 0; a.out_scale = 1.0f;
  a.geo = make_geo(n_in, C, pos_emb);
  UttPlan u;
  if (int rc = utterance_run_plan(a.geo, sv, precision, kUttValidate, workspace_bytes, who, &u)) return rc;
  a.loss_partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + u.part_off);
  return launch_utterances(a, u, sv, workspace, seg_loss_out, loss_out, (cudaStream_t)stream);
}

extern "C" int b2h_train_step_dp(const void* x, int x_dtype, const float* target, const float* conf, const int32_t* lengths,
                                 float* params, void* packed, float* exp_avg, float* exp_avg_sq, float* loss_out, int B, int T,
                                 int n_in, int C, int pos_emb, int loss_kind, int precision, double lr, double beta1,
                                 double beta2, double eps, int64_t* step_dev, int64_t* epoch_dev, const double* lr_dev,
                                 float* sym_grads, const void* peer_bufs_dev, void* multicast_buf, int rank, int world,
                                 float grad_scale, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!exp_avg || !exp_avg_sq || !loss_out || !step_dev || !epoch_dev || !sym_grads || !peer_bufs_dev) {
    set_error("b2h_train_step_dp: null pointer");
    return B2H_EINVAL;
  }
  if (world < 1 || world > 32 || rank < 0 || rank >= world) { set_error("b2h_train_step_dp: bad rank/world"); return B2H_EINVAL; }
  FuseAdam fuse = fuse_adam(params, packed, exp_avg, exp_avg_sq, loss_out, lr, beta1, beta2, eps, grad_scale, step_dev, lr_dev);
  fuse.peer_bufs = reinterpret_cast<const float* const*>(peer_bufs_dev); fuse.sym_grads = sym_grads;
  fuse.mc_buf = reinterpret_cast<unsigned long long*>(multicast_buf);
  fuse.epoch_dev = reinterpret_cast<const long long*>(epoch_dev); fuse.rank = rank; fuse.world = world;
  const TrainResult r = train_common(x, x_dtype, nullptr, nullptr, target, conf, nullptr, lengths, params, packed, nullptr, B, T,
                                     n_in, C, pos_emb, loss_kind, precision, 1, workspace, workspace_bytes, (cudaStream_t)stream,
                                     "b2h_train_step_dp", reinterpret_cast<long long*>(step_dev),
                                     reinterpret_cast<long long*>(epoch_dev), &fuse);
  if (r.rc) return r.rc;
  if (r.plan.kernel == B2H_KERNEL_TC_TILE) return B2H_OK;    // everything happened inside the one cooperative launch
  if (int rc = launch_reduce(r.partials, r.plan.nparts, r.g, sym_grads, r.loss_partials, r.plan.n_loss, loss_out,
                             reinterpret_cast<const long long*>(epoch_dev), (cudaStream_t)stream))
    return rc;
  return launch_adam_dp(params, reinterpret_cast<const float* const*>(peer_bufs_dev), rank, world, exp_avg, exp_avg_sq, r.g.P, lr,
                        beta1, beta2, eps, reinterpret_cast<const long long*>(step_dev),
                        reinterpret_cast<const long long*>(epoch_dev), lr_dev, grad_scale, packed, r.g, (cudaStream_t)stream);
}

extern "C" int b2h_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, double lr,
                             double beta1, double beta2, double eps, int64_t step, const int64_t* step_dev,
                             const double* lr_dev, float grad_scale, void* packed, int n_in, int C, int pos_emb, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq) { set_error("b2h_adam_step: null pointer"); return B2H_EINVAL; }
  if ((step < 1 && !step_dev) || n < 0) { set_error("b2h_adam_step: bad step/n"); return B2H_EINVAL; }
  Geo g{};
  if (packed) {
    if (!geo_ok(n_in, C, pos_emb, "b2h_adam_step")) return B2H_ESHAPE;
    g = make_geo(n_in, C, pos_emb);
    if (g.P != n) { set_error("b2h_adam_step: n=%lld does not match geometry (%d)", (long long)n, g.P); return B2H_ESHAPE; }
  }
  if (n == 0) return B2H_OK;
  return launch_adam_flat(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step < 1 ? 1 : step,
                          reinterpret_cast<const long long*>(step_dev), lr_dev, grad_scale, packed, g, (cudaStream_t)stream);
}

extern "C" int b2h_mask_output(float* y, const int32_t* lengths, int B, int T, int row_elems, void* stream) {
  if (!y || !lengths) { set_error("b2h_mask_output: null pointer"); return B2H_EINVAL; }
  if (B < 0 || T < 0 || row_elems < 1) { set_error("b2h_mask_output: bad shape"); return B2H_ESHAPE; }
  return launch_mask_output(y, lengths, B, T, row_elems, (cudaStream_t)stream);
}

extern "C" int b2h_pose_l1(const float* pred, const float* target, const float* scores, const int32_t* lengths, int B, int T,
                           int row_elems, int loss_kind, float* loss_out, float* d_pred, float* row_scratch, void* stream) {
  if (!pred || !target || !lengths || !loss_out || !row_scratch) { set_error("b2h_pose_l1: null pointer"); return B2H_EINVAL; }
  if (loss_kind != B2H_LOSS_L1 && loss_kind != B2H_LOSS_CONFL1) { set_error("b2h_pose_l1: bad loss_kind"); return B2H_EINVAL; }
  if (loss_kind == B2H_LOSS_CONFL1 && (!scores || (row_elems & 1))) { set_error("b2h_pose_l1: confL1 needs scores and even row_elems"); return B2H_EINVAL; }
  if (B < 1 || T < 1 || row_elems < 1) { set_error("b2h_pose_l1: bad shape"); return B2H_ESHAPE; }
  return launch_pose_l1(pred, target, scores, lengths, B, T, row_elems, loss_kind, loss_out, d_pred, row_scratch, (cudaStream_t)stream);
}

extern "C" int b2h_format_prediction(const float* pred, float* out, int64_t rows, int mode, void* stream) {
  if (!pred || !out) { set_error("b2h_format_prediction: null pointer"); return B2H_EINVAL; }
  if (rows < 0 || (mode != 0 && mode != 1)) { set_error("b2h_format_prediction: bad rows/mode"); return B2H_EINVAL; }
  return launch_format_prediction(pred, out, rows, mode, (cudaStream_t)stream);
}

extern "C" int b2h_pos_emb_concat(const float* inp, float* out, int B, int channels, int T, int max_len, void* stream) {
  if (!inp || !out) { set_error("b2h_pos_emb_concat: null pointer"); return B2H_EINVAL; }
  if (B < 0 || channels < 1 || T < 1 || max_len < 1) { set_error("b2h_pos_emb_concat: bad shape"); return B2H_ESHAPE; }
  if (T != max_len) {   // torch.cat of (B,1,max_len) with (B,C,T) fails in the reference (HandPoseModels.py:82)
    set_error("b2h_pos_emb_concat: Sizes of tensors must match except in dimension 1 (T=%d, max_len=%d)", T, max_len);
    return B2H_ESHAPE;
  }
  return launch_pos_emb_concat(inp, out, B, channels, T, max_len, (cudaStream_t)stream);
}

extern "C" int b2h_tc_probe(const void* a_bf16, const void* b_bf16, float* out, int n, int ksteps, int shift, int variant,
                            void* stream) {
  if (!a_bf16 || !b_bf16 || !out) { set_error("b2h_tc_probe: null pointer"); return B2H_EINVAL; }
  return launch_tc_probe(a_bf16, b_bf16, out, n, ksteps, shift, variant, (cudaStream_t)stream);
}

extern "C" void b2h_debug_timing(void* dev_i64x1024) { set_debug_timing(reinterpret_cast<long long*>(dev_i64x1024)); }

extern "C" int b2h_tc_status(void) { return tc_status_and_clear(); }

namespace {
constexpr int kMaxDev = 64;
std::mutex g_cache_mu;
int g_sms[kMaxDev] = {0};
struct SmemAttr { const void* fn; size_t bytes[kMaxDev]; };
SmemAttr g_attr[32] = {};
int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; }
  return dev < 0 ? 0 : dev;
}
}  // namespace

int b2h::num_sms() {
  const int dev = current_device();
  std::lock_guard<std::mutex> lk(g_cache_mu);
  if (dev < kMaxDev && g_sms[dev]) return g_sms[dev];
  int n = 0;
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (n <= 0) n = 148;
  if (dev < kMaxDev) g_sms[dev] = n;
  return n;
}

int b2h::ensure_dyn_smem(const void* fn, size_t bytes) {
  const int dev = current_device();
  std::lock_guard<std::mutex> lk(g_cache_mu);
  SmemAttr* slot = nullptr;
  for (auto& a : g_attr) {
    if (a.fn == fn) { slot = &a; break; }
    if (!a.fn) { a.fn = fn; slot = &a; break; }
  }
  if (slot && dev < kMaxDev && slot->bytes[dev] >= bytes) return B2H_OK;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaFuncSetAttribute(%zu B): %s", bytes, cudaGetErrorString(e)); return B2H_ECUDA; }
  if (slot && dev < kMaxDev) slot->bytes[dev] = bytes;
  return B2H_OK;
}
