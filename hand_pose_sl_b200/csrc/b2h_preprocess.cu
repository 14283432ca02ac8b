// K0 -- keypoint preprocessing: 12-of-25 gather, xy/conf split, crop/pad windowing,
// wrist/neck-relative differencing, /1280 normalisation.  HBM-bound, bit-exact.
//
// Reference semantics (paths relative to the reference root):
//   load_keypoints / BODY_HEAD_KEYPOINTS     body2hand/src/dataloaders/text_pose_dataset.py:14-50
//   select_jsons crop, pad, clip, n_frames   ...text_pose_dataset.py:52-68, 447, 511-529, 614-635
//   WristDifference / ChestDifference        body2hand/src/steps/utils.py:194-210
//   NormalizeFixedFactor                     body2hand/src/steps/utils.py:180-190
//   BuildRightHandItem                       body2hand/src/steps/utils.py:261-277
//   TextPoseH5Dataset.array2item             ...text_pose_dataset.py:587-612
//
// Design: one warp owns 4 consecutive window slots.  4 OpenPose frames are 1200 B (pose) + 2 x 1008 B (hands): all three
// are 16-B multiples, so an aligned 4-frame group travels HBM -> shared memory as three TMA bulk copies into the warp's
// double buffer, one group ahead of the compute (mbarrier completion).  The wrist / neck references are shared through
// the staged tile; a per-CTA gather table says where every output element's source and reference sit, and the six output
// rows of the 4 slots (162 float4) go back with coalesced 128-bit streaming stores.  Padded / unaligned groups are filled
// by the lanes inside the same kernel (warp-uniform branch).  IEEE sub.rn then div.rn: no reciprocal shortcut that is not
// verified bit-exact, no FMA contraction across the two.
#include "b2h_common.cuh"
#define B2H_TC_NO_STATUS
#include "b2h_tc.cuh"   // mbarrier + 1-D TMA bulk copy helpers

namespace b2h {

constexpr int kWarpsPerBlock = 6;      // the per-CTA gather table (162 float4 slots, one per thread) is built once for 6 warps
constexpr int kBlocksPerSM = 4;        // 4 x 41.5 KB of static shared memory; 24 warps and 77 KB of bulk copies in flight per SM
// set when a wait for a staged 4-frame group (TMA bulk copy) exceeded its ~2 s budget: the launch's outputs are then
// incomplete; read and cleared by b2h_preprocess_status()
__device__ int g_pre_status = 0;

template <int FMT> struct Fmt;
// FMT 0: OpenPose [x,y,c] rows: pose25 (75) | hand_left (63) | hand_right (63)
template <> struct Fmt<0> {
  static constexpr int kBody = 12;
  static constexpr int kSrc = 3;
  static constexpr int kStage = 4 * (75 + 63 + 63);  // 804 floats per warp
  __device__ static int src_len(int a) { return a == 0 ? 75 : 63; }
  __device__ static int src_off(int a) { return a == 0 ? 0 : (a == 1 ? 300 : 552); }
  __device__ static int body_idx(int j) { return j < 8 ? j : j + 7; }  // BODY_HEAD_KEYPOINTS
  __device__ static const float& body_ref(const float* st, int i, int j, int d) { return st[i * 75 + 3 * body_idx(j) + d]; }
  __device__ static const float& lh_ref(const float* st, int i, int j, int d) { return st[300 + i * 63 + 3 * j + d]; }
  __device__ static const float& rh_ref(const float* st, int i, int j, int d) { return st[552 + i * 63 + 3 * j + d]; }
  __device__ static float body(const float* st, int i, int j, int d) { return st[i * 75 + 3 * body_idx(j) + d]; }
  __device__ static float lh(const float* st, int i, int j, int d) { return st[300 + i * 63 + 3 * j + d]; }
  __device__ static float rh(const float* st, int i, int j, int d) { return st[552 + i * 63 + 3 * j + d]; }
};
// FMT 1: packed H5 rows (150) = [x0..x49 | y0..y49 | c0..c49]; body 0..7, left hand 8..28, right 29..49
template <> struct Fmt<1> {
  static constexpr int kBody = 8;
  static constexpr int kSrc = 1;
  static constexpr int kStage = 4 * 150;
  __device__ static int src_len(int) { return 150; }
  __device__ static int src_off(int) { return 0; }
  __device__ static const float& body_ref(const float* st, int i, int j, int d) { return st[i * 150 + d * 50 + j]; }
  __device__ static const float& lh_ref(const float* st, int i, int j, int d) { return st[i * 150 + d * 50 + 8 + j]; }
  __device__ static const float& rh_ref(const float* st, int i, int j, int d) { return st[i * 150 + d * 50 + 29 + j]; }
  __device__ static float body(const float* st, int i, int j, int d) { return st[i * 150 + d * 50 + j]; }
  __device__ static float lh(const float* st, int i, int j, int d) { return st[i * 150 + d * 50 + 8 + j]; }
  __device__ static float rh(const float* st, int i, int j, int d) { return st[i * 150 + d * 50 + 29 + j]; }
};

struct PreArgs {
  const float* src[3];
  int64_t n_frames;
  const int64_t* win_start;
  const int64_t* win_end;   // nullable: exclusive end of the clip each window is cropped from (default n_frames)
  int n_win, T, pad_mode, dif, normalize, aligned, fastdiv;
  float factor, rfactor;
  float* out[6];  // input_kp, input_conf, target_kp, target_conf, left_kp, left_conf
  int64_t* n_frames_out;
  __nv_bfloat16* input_bf16;
};

// Exact division by the normalisation factor without the generic div.rn sequence (whose special-operand
// slow path is taken for every zero = undetected keypoint).  With rc = RN(1/c):  q = RN(x*rc),
// r = x - q*c (exact, FMA), q' = RN(q + r*rc) is the correctly rounded x/c (Markstein) as long as nothing
// over/underflows (x = 0, or 1e-30 < |x| < 1e30); outside that range the IEEE routine is used.  tests/test_gpu_preprocess.py checks the
// identity for c = 1280 over ALL 2^32 float bit patterns on the device (b2h_verify_fastdiv).
// The range test works on the magnitude bits: (u - 1) wraps u = 0 to the top, so "u - 1 >= lo" reads "zero, or above lo".
constexpr uint32_t kDivLo = 0x0DA24260u;   // bits of 1e-30f
constexpr uint32_t kDivHi = 0x7149F2CAu;   // bits of 1e30f
__device__ __forceinline__ bool div_in_range(float x) {
  const uint32_t u = __float_as_uint(x) & 0x7FFFFFFFu;
  return u < kDivHi && (u - 1u) >= kDivLo;
}
// valid when div_in_range(x); the quotient carries x's sign (c > 0), which also restores -0 (the FMA chain returns +0)
__device__ __forceinline__ float div_fast(float x, float c, float rc) {
  const float q = __fmul_rn(x, rc);
  const float r = __fmaf_rn(-q, c, x);
  const float res = __fmaf_rn(r, rc, q);
  return __uint_as_float((__float_as_uint(res) & 0x7FFFFFFFu) | (__float_as_uint(x) & 0x80000000u));
}
__device__ __forceinline__ float div_exact(float x, float c, float rc) {
  return div_in_range(x) ? div_fast(x, c, rc) : __fdiv_rn(x, c);   // the IEEE routine is never taken on keypoint data
}
// four quotients, one range test: all four magnitudes through an unsigned max / a wrapped unsigned min
__device__ __forceinline__ void div_exact4(float (&v)[4], float c, float rc) {
  uint32_t mx = 0u, mn = 0xFFFFFFFFu;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const uint32_t u = __float_as_uint(v[e]) & 0x7FFFFFFFu;
    mx = max(mx, u);
    mn = min(mn, u - 1u);
  }
  if (mx < kDivHi && mn >= kDivLo) {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = div_fast(v[e], c, rc);
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = __fdiv_rn(v[e], c);
  }
}

template <int FMT>
__device__ __forceinline__ float out_elem(const float* st, int a, int i, int r, const PreArgs& p) {
  using F = Fmt<FMT>;
  float v;
  switch (a) {
    case 0: {  // input_kp = (body - neck) / factor          utils.py:209, :186, :265
      int j = r >> 1, d = r & 1;
      v = F::body(st, i, j, d);
      if (p.dif) v = __fsub_rn(v, F::body(st, i, 1, d));
      if (p.normalize) v = p.fastdiv ? div_exact(v, p.factor, p.rfactor) : __fdiv_rn(v, p.factor);
      return v;
    }
    case 1: return F::body(st, i, r, 2);  // input_conf     utils.py:268
    case 2: {  // target_kp = (right_hand - raw right wrist) / factor   utils.py:200, :187, :266
      int j = r >> 1, d = r & 1;
      v = F::rh(st, i, j, d);
      if (p.dif) v = __fsub_rn(v, F::body(st, i, 4, d));
      if (p.normalize) v = __fdiv_rn(v, p.factor);
      return v;
    }
    case 3: return F::rh(st, i, r, 2);    // target_conf    utils.py:269
    case 4: {  // left hand is only scaled, never differenced    utils.py:188
      int j = r >> 1, d = r & 1;
      v = F::lh(st, i, j, d);
      if (p.normalize) v = __fdiv_rn(v, p.factor);
      return v;
    }
    default: return F::lh(st, i, r, 2);
  }
}

__global__ void verify_fastdiv_kernel(float c, float rc, unsigned long long* mismatches) {
  unsigned long long bad = 0;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32);
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const float x = __uint_as_float((unsigned)i);
    const float a = div_exact(x, c, rc), b = __fdiv_rn(x, c);
    const bool same = (__float_as_uint(a) == __float_as_uint(b)) || (a != a && b != b);
    bad += same ? 0 : 1;
  }
  if (bad) atomicAdd(mismatches, bad);
}

// Gather table (built once per CTA in shared memory): for every output float4 of a 4-slot group, which array
// it belongs to and, per element, where its source value and its reference (neck / wrist, or a zero slot)
// sit in the staged tile.  The keypoint arrays (difference [+ division]) come first, the confidences (plain gather) after
// them, and each kind has its own rounds, so the steady-state loop has no per-element flags:
// 2 x LDS.128 (offsets) + 8 LDS + 4 sub.rn [+ exact division] + STG.128 per keypoint float4, LDS.128 + 4 LDS + STG.128
// per confidence float4.        qinfo: bits 0-7 float4 index in the array block, 8-10 array
template <int FMT, int A>
__device__ __forceinline__ void table_entry(int i, int r, int dif, int zero_slot, uint32_t& src_b, uint32_t& ref_b) {
  using F = Fmt<FMT>;
  const float* z = nullptr;
  uint32_t src = 0, ref = (uint32_t)zero_slot;
  const int j = r >> 1, d = r & 1;
  if (A == 0) { src = (uint32_t)(&F::body_ref(z, i, j, d) - z); if (dif) ref = (uint32_t)(&F::body_ref(z, i, 1, d) - z); }
  else if (A == 1) src = (uint32_t)(&F::body_ref(z, i, r, 2) - z);
  else if (A == 2) { src = (uint32_t)(&F::rh_ref(z, i, j, d) - z); if (dif) ref = (uint32_t)(&F::body_ref(z, i, 4, d) - z); }
  else if (A == 3) src = (uint32_t)(&F::rh_ref(z, i, r, 2) - z);
  else if (A == 4) src = (uint32_t)(&F::lh_ref(z, i, j, d) - z);
  else src = (uint32_t)(&F::lh_ref(z, i, r, 2) - z);
  src_b = src * 4u; ref_b = ref * 4u;            // byte offsets into the warp's staged tile
}

// one array's share of the gather table: its float4 slots are [base, base + N); N (floats per frame = float4 per 4-slot
// group) is a compile-time constant, so the slot -> (frame, element) split is a multiply-shift
template <int FMT, int A, int N>
__device__ __forceinline__ void build_array(int q, int base, int dif, int zero_slot, uint32_t* tab_src, uint32_t* tab_ref,
                                            uint16_t* qinfo) {
  const int ql = q - base;
  if (ql < 0 || ql >= N) return;
  qinfo[q] = (uint16_t)(ql | (A << 8));
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int idx = ql * 4 + e;
    const int i = idx / N, r = idx - i * N;
    uint32_t sb, rb;
    table_entry<FMT, A>(i, r, dif, zero_slot, sb, rb);
    tab_src[q * 4 + e] = sb;
    if ((A & 1) == 0) tab_ref[q * 4 + e] = rb;   // keypoint arrays come first: their slots index tab_ref directly
  }
}

template <int FMT>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, kBlocksPerSM) preprocess_kernel(PreArgs p) {
  using F = Fmt<FMT>;
  constexpr int kMaxQ = F::kBody * 3 + 126;             // float4 per 4-slot group over all six arrays
  constexpr int kZero = F::kStage;                      // 4 zero floats behind every warp's staged tile
  static_assert(kMaxQ <= kWarpsPerBlock * 32, "the table build gives every float4 slot its own thread");
  __shared__ __align__(16) float stage_all[kWarpsPerBlock][2][F::kStage + 4];   // double-buffered per warp
  __shared__ __align__(8) uint64_t sbar[kWarpsPerBlock][2];
  constexpr int kMaxKp = F::kBody * 2 + 84;             // float4 per group over the three keypoint arrays
  __shared__ __align__(16) uint32_t tab_src[kMaxQ * 4];
  __shared__ __align__(16) uint32_t tab_ref[kMaxKp * 4];
  __shared__ uint16_t qinfo[kMaxQ];
  __shared__ float* s_out[6];
  __shared__ int s_nq, s_nkp;
  const int lane = threadIdx.x & 31;
  const int wib = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);     // warp-uniform (uniform-register addressing of the tile)
  const int64_t S = (int64_t)p.n_win * p.T;
  const int64_t n_groups = (S + 3) >> 2;
  const bool small = S < (int64_t)0x7fffffff;
  // each warp owns its two staging buffers and their barriers: no CTA-wide sync is needed before its first copy
  if (lane < 8) stage_all[wib][lane >> 2][kZero + (lane & 3)] = 0.0f;
  if (lane == 0) { tc::mbar_init(&sbar[wib][0], 1); tc::mbar_init(&sbar[wib][1], 1); tc::fence_barrier_init(); }
  __syncwarp();

  // Stage the 4 source frames of group gg into buffer b of this warp.  Aligned groups are moved by the TMA engine
  // (3 bulk copies, completion on the buffer's mbarrier) one group AHEAD of the compute; padded / unaligned groups
  // are filled by the lanes.  Either way exactly one arrival completes the buffer's phase.
  auto issue = [&](int64_t gg, int b) {
    float* st = stage_all[wib][b];
    const int64_t s0 = gg << 2;
    // window index math (bit-exact integer work): slot s -> (window, t) -> source frame
    int64_t w; int t;
    if (small) { const int si = (int)s0; const int wi = si / p.T; w = wi; t = si - wi * p.T; }
    else { w = s0 / p.T; t = (int)(s0 - w * p.T); }
    auto bulk = [&](int64_t f0) {                    // 4 consecutive, 16-B aligned source frames: the TMA engine moves them
      if (lane == 0) {
        uint32_t bytes = 0;
#pragma unroll
        for (int a = 0; a < F::kSrc; ++a) bytes += 16u * F::src_len(a);
        tc::mbar_arrive_expect_tx(&sbar[wib][b], bytes);
#pragma unroll
        for (int a = 0; a < F::kSrc; ++a)
          tc::bulk_g2s(st + F::src_off(a), p.src[a] + f0 * F::src_len(a), 16u * F::src_len(a), &sbar[wib][b]);
      }
    };
    // Common case first: the 4 slots lie in ONE window and inside its clip -- one crop, no pad rule.  Same integer
    // results as the per-slot walk below (f_i = start + t + i, all inside [0, cend)).
    if (p.aligned && t + 3 < p.T && s0 + 3 < S) {
      const int64_t start = p.win_start[w];
      int64_t cend = p.win_end ? p.win_end[w] : p.n_frames;
      cend = cend > p.n_frames ? p.n_frames : cend;
      const int64_t f0 = start + t;
      if (f0 >= 0 && f0 + 3 < cend && (f0 & 3) == 0) {
        if (t == 0 && lane == 0 && p.n_frames_out) {
          const int64_t rem = cend - start;
          p.n_frames_out[w] = rem < p.T ? rem : (int64_t)p.T;   // :447 (rem >= 4 here)
        }
        bulk(f0);
        return;
      }
    }
    int64_t srcf[4];
    bool consecutive = true;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (s0 + i < S) {
        const int64_t start = p.win_start[w];
        int64_t cend = p.win_end ? p.win_end[w] : p.n_frames;      // end of the utterance this window belongs to
        cend = cend > p.n_frames ? p.n_frames : cend;
        int64_t f = start + t;                        // crop [start, start+T)   text_pose_dataset.py:66-68
        if (f >= cend || f < 0)                       // past the clip end -> pad rule
          f = (p.pad_mode == B2H_PAD_REPEAT_FIRST && start >= 0 && start < cend) ? start : -1;  // :512-518 / :616-622
        srcf[i] = f;
        if (t == 0 && lane == 0 && p.n_frames_out) {
          const int64_t rem = cend - start;
          p.n_frames_out[w] = rem < 0 ? 0 : (rem < p.T ? rem : (int64_t)p.T);   // :447
        }
      } else {
        srcf[i] = -1;
      }
      if (i > 0 && srcf[i] != srcf[0] + i) consecutive = false;
      if (++t == p.T) { t = 0; ++w; }
    }
    const bool fast = p.aligned && consecutive && srcf[0] >= 0 && (srcf[0] & 3) == 0 && (s0 + 3 < S);
    if (fast) {
      bulk(srcf[0]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int a = 0; a < F::kSrc; ++a) {
          const int len = F::src_len(a);
          float* sdst = st + F::src_off(a) + i * len;
          if (srcf[i] >= 0) {
            const float* gsrc = p.src[a] + srcf[i] * len;
            for (int q = lane; q < len; q += 32) sdst[q] = __ldcs(gsrc + q);
          } else {
            for (int q = lane; q < len; q += 32) sdst[q] = 0.0f;
          }
        }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&sbar[wib][b]);
    }
  };

  const int64_t gstride = (int64_t)gridDim.x * kWarpsPerBlock;
  int64_t g = (int64_t)blockIdx.x * kWarpsPerBlock + wib;
  if (g < n_groups) issue(g, 0);      // the first group travels while the CTA builds its gather table

  // ---- build the gather table: divided arrays (keypoints) first, then pass-through arrays (confidences) ----
  {
    constexpr int kB = F::kBody;
    const int q = threadIdx.x;                          // kMaxQ <= blockDim.x: one float4 slot per thread
    int acc = 0;
    if (p.out[0]) { build_array<FMT, 0, 2 * kB>(q, acc, p.dif, kZero, tab_src, tab_ref, qinfo); acc += 2 * kB; }
    if (p.out[2]) { build_array<FMT, 2, 42>(q, acc, p.dif, kZero, tab_src, tab_ref, qinfo); acc += 42; }
    if (p.out[4]) { build_array<FMT, 4, 42>(q, acc, p.dif, kZero, tab_src, tab_ref, qinfo); acc += 42; }
    const int nkp_ = acc;
    if (p.out[1]) { build_array<FMT, 1, kB>(q, acc, p.dif, kZero, tab_src, tab_ref, qinfo); acc += kB; }
    if (p.out[3]) { build_array<FMT, 3, 21>(q, acc, p.dif, kZero, tab_src, tab_ref, qinfo); acc += 21; }
    if (p.out[5]) { build_array<FMT, 5, 21>(q, acc, p.dif, kZero, tab_src, tab_ref, qinfo); acc += 21; }
    if (threadIdx.x == 0) {
      s_nq = acc; s_nkp = nkp_;
#pragma unroll
      for (int a = 0; a < 6; ++a) s_out[a] = p.out[a];
    }
  }
  __syncthreads();
  const int nq = s_nq, nkp = s_nkp;
  const float factor = p.factor, rfactor = p.rfactor;
  const bool fastdiv = p.fastdiv != 0, normalize = p.normalize != 0;
  // Every lane owns the same output float4 slots (q = lane + 32*round) in every group, so its destination array
  // and row length are loop invariants kept in registers.
  constexpr int kKpRounds = (kMaxKp + 31) / 32, kConfRounds = (kMaxQ - kMaxKp + 31) / 32;
  float* okp[kKpRounds];
  float* ocf[kConfRounds];
  int nkp_row[kKpRounds], ncf_row[kConfRounds];
  auto slot_dest = [&](int q, float*& ob, int& n) {     // destination of float4 slot q in slot-group 0, floats per frame
    const int qi = qinfo[q];
    const int a = qi >> 8;
    n = (a == 0) ? F::kBody * 2 : (a == 1) ? F::kBody : ((a & 1) ? 21 : 42);
    ob = s_out[a] + (qi & 255) * 4;
  };
#pragma unroll
  for (int r = 0; r < kKpRounds; ++r) {
    okp[r] = nullptr; nkp_row[r] = 0;
    if (lane + 32 * r < nkp) slot_dest(lane + 32 * r, okp[r], nkp_row[r]);
  }
#pragma unroll
  for (int r = 0; r < kConfRounds; ++r) {
    ocf[r] = nullptr; ncf_row[r] = 0;
    if (nkp + lane + 32 * r < nq) slot_dest(nkp + lane + 32 * r, ocf[r], ncf_row[r]);
  }

  for (int it = 0; g < n_groups; g += gstride, ++it) {
    const int b = it & 1;
    __syncwarp();                                   // every lane is done reading buffer b^1 (previous group)
    if (g + gstride < n_groups) issue(g + gstride, b ^ 1);
    {                                               // wait for this group's frames
      const uint32_t parity = (uint32_t)(it >> 1) & 1u;
      const long long t0 = clock64();
      while (!tc::mbar_try_wait(&sbar[wib][b], parity))
        if (clock64() - t0 > 4000000000LL) {        // never spin forever: record the failure (b2h_preprocess_status) and go on
          atomicExch(&g_pre_status, 1);
          break;
        }
    }
    const float* st = stage_all[wib][b];
    const char* stb = reinterpret_cast<const char*>(st);
    const int64_t s0 = g << 2;
    const bool full = (s0 + 3 < S);
    // ---- the six output rows of the 4 slots ----
    if (full) {
#pragma unroll
      for (int r = 0; r < kKpRounds; ++r) {            // keypoints: utils.py:200 / :209 (x - 0 = x when there is no reference)
        const int q = lane + 32 * r;
        if (q < nkp) {
          const uint4 s4 = *reinterpret_cast<const uint4*>(tab_src + q * 4);
          const uint4 r4 = *reinterpret_cast<const uint4*>(tab_ref + q * 4);
          const uint32_t so[4] = {s4.x, s4.y, s4.z, s4.w}, ro[4] = {r4.x, r4.y, r4.z, r4.w};
          float v[4];
#pragma unroll
          for (int e = 0; e < 4; ++e)
            v[e] = __fsub_rn(*reinterpret_cast<const float*>(stb + so[e]), *reinterpret_cast<const float*>(stb + ro[e]));
          if (normalize) {                                                                   // utils.py:186-188
            if (fastdiv) {
              div_exact4(v, factor, rfactor);
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e) v[e] = __fdiv_rn(v[e], factor);
            }
          }
          __stcs(reinterpret_cast<float4*>(okp[r] + s0 * nkp_row[r]), make_float4(v[0], v[1], v[2], v[3]));
        }
      }
#pragma unroll
      for (int r = 0; r < kConfRounds; ++r) {          // confidences: plain gather   utils.py:268-269
        const int q = nkp + lane + 32 * r;
        if (q < nq) {
          const uint4 s4 = *reinterpret_cast<const uint4*>(tab_src + q * 4);
          const float4 v = make_float4(*reinterpret_cast<const float*>(stb + s4.x), *reinterpret_cast<const float*>(stb + s4.y),
                                       *reinterpret_cast<const float*>(stb + s4.z), *reinterpret_cast<const float*>(stb + s4.w));
          __stcs(reinterpret_cast<float4*>(ocf[r] + s0 * ncf_row[r]), v);
        }
      }
      if (p.input_bf16) {  // bf16 copy of input_kp for the tensor-core net (no second pass over HBM)
        const int n = F::kBody * 2;
        for (int q = lane; q < n / 2; q += 32) {      // n*4 bf16 = n/2 x 16-B chunks
          __nv_bfloat16 h[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            int idx = q * 8 + e;
            int i = idx / n, r = idx - i * n;
            h[e] = __float2bfloat16_rn(out_elem<FMT>(st, 0, i, r, p));
          }
          reinterpret_cast<uint4*>(p.input_bf16 + s0 * n)[q] = *reinterpret_cast<uint4*>(h);
        }
      }
    } else {  // ragged tail (S % 4 != 0): scalar stores
      const int nvalid = (int)(S - s0);
      for (int a = 0; a < 6; ++a) {
        if (p.out[a] == nullptr) continue;
        const int n = (a == 0) ? F::kBody * 2 : (a == 1) ? F::kBody : ((a & 1) ? 21 : 42);
        for (int idx = lane; idx < nvalid * n; idx += 32) {
          int i = idx / n, r = idx - i * n;
          p.out[a][s0 * n + idx] = out_elem<FMT>(st, a, i, r, p);
        }
      }
      if (p.input_bf16) {
        const int n = F::kBody * 2;
        for (int idx = lane; idx < nvalid * n; idx += 32) {
          int i = idx / n, r = idx - i * n;
          p.input_bf16[s0 * n + idx] = __float2bfloat16_rn(out_elem<FMT>(st, 0, i, r, p));
        }
      }
    }
  }
}

template <int FMT>
static int launch_pre(PreArgs& p, cudaStream_t stream) {
  if (p.n_win <= 0 || p.T <= 0) return B2H_OK;
  int64_t S = (int64_t)p.n_win * p.T;
  int64_t groups = (S + 3) / 4;
  int64_t blocks = (groups + kWarpsPerBlock - 1) / kWarpsPerBlock;
  // Resident CTAs, grid-stride beyond that.  Measured on B200 (profiles/r2_k0_residency.txt): while the launch's bytes fit
  // the 126 MB L2 with room to spare, 4 CTAs/SM (24 warps) are fastest (1 h clip: 28.1 vs 31.0 us); once reads and writes
  // both stream through DRAM, 2 CTAs/SM keep fewer DRAM pages open at a time and win (2 h: 56.8 vs 60.6 us, 8 h: 209 vs
  // 236 us = 0.92 of the measured copy peak).
  using F = Fmt<FMT>;
  const int out_floats[6] = {F::kBody * 2, F::kBody, 42, 21, 42, 21};
  int64_t bytes_per_slot = (FMT == 0 ? 804 : 600) + (p.input_bf16 ? F::kBody * 4 : 0);
  for (int a = 0; a < 6; ++a) bytes_per_slot += p.out[a] ? out_floats[a] * 4 : 0;
  const int per_sm = S * bytes_per_slot > (int64_t)190 * 1000 * 1000 ? 2 : kBlocksPerSM;
  int64_t cap = (int64_t)num_sms() * per_sm;
  if (blocks > cap) blocks = cap;
  preprocess_kernel<FMT><<<(unsigned)blocks, kWarpsPerBlock * 32, 0, stream>>>(p);
  count_launch();
  return check_launch("preprocess_kernel");
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace b2h

using namespace b2h;

extern "C" int b2h_preprocess_status(void) {
  int v = 0, z = 0;
  cudaMemcpyFromSymbol(&v, g_pre_status, sizeof(int));
  if (v) cudaMemcpyToSymbol(g_pre_status, &z, sizeof(int));
  return v;
}

extern "C" int b2h_verify_fastdiv(float factor, unsigned long long* mismatches_dev, void* stream) {
  if (!mismatches_dev) { set_error("b2h_verify_fastdiv: null pointer"); return B2H_EINVAL; }
  verify_fastdiv_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(factor, 1.0f / factor, mismatches_dev);
  count_launch();
  return check_launch("verify_fastdiv_kernel");
}

extern "C" int b2h_preprocess(const float* pose25, const float* hand_left, const float* hand_right, int64_t n_frames,
                              const int64_t* win_start, const int64_t* win_end, int n_win, int T, int pad_mode, float factor,
                              int dif_encoding, int normalize, float* input_kp, float* input_conf,
                              float* target_kp, float* target_conf, float* left_kp, float* left_conf,
                              int64_t* n_frames_out, void* input_kp_bf16, void* stream) {
  if (!pose25 || !hand_left || !hand_right || !win_start) { set_error("b2h_preprocess: null pointer"); return B2H_EINVAL; }
  if (!input_kp && !input_conf && !target_kp && !target_conf && !left_kp && !left_conf && !input_kp_bf16) {
    set_error("b2h_preprocess: no output requested");
    return B2H_EINVAL;
  }
  if (pad_mode != B2H_PAD_REPEAT_FIRST && pad_mode != B2H_PAD_ZEROS) { set_error("b2h_preprocess: bad pad_mode %d", pad_mode); return B2H_EINVAL; }
  if (n_frames < 0 || n_win < 0 || T < 0) { set_error("b2h_preprocess: negative size"); return B2H_ESHAPE; }
  PreArgs p{};
  p.src[0] = pose25; p.src[1] = hand_left; p.src[2] = hand_right;
  p.n_frames = n_frames; p.win_start = win_start; p.win_end = win_end; p.n_win = n_win; p.T = T; p.pad_mode = pad_mode;
  p.dif = dif_encoding; p.normalize = normalize; p.factor = factor;
  p.rfactor = 1.0f / factor; p.fastdiv = (factor == 1280.0f) ? 1 : 0;   // the reference's factor (run.py:90): verified exhaustively
  p.out[0] = input_kp; p.out[1] = input_conf; p.out[2] = target_kp; p.out[3] = target_conf;
  p.out[4] = left_kp; p.out[5] = left_conf;
  p.n_frames_out = n_frames_out; p.input_bf16 = reinterpret_cast<__nv_bfloat16*>(input_kp_bf16);
  bool al = aligned16(pose25) && aligned16(hand_left) && aligned16(hand_right) && aligned16(input_kp_bf16);
  for (int a = 0; a < 6; ++a) al = al && aligned16(p.out[a]);
  if (!al) { set_error("b2h_preprocess: pointers must be 16-byte aligned"); return B2H_EALIGN; }
  p.aligned = 1;
  return launch_pre<0>(p, (cudaStream_t)stream);
}

extern "C" int b2h_preprocess_h5(const float* rows150, int64_t n_frames, const int64_t* win_start, const int64_t* win_end,
                                 int n_win, int T,
                                 int pad_mode, float factor, int dif_encoding, int normalize, float* input_kp,
                                 float* input_conf, float* target_kp, float* target_conf, float* left_kp,
                                 float* left_conf, int64_t* n_frames_out, void* stream) {
  if (!rows150 || !win_start || !input_kp || !input_conf || !target_kp || !target_conf) {
    set_error("b2h_preprocess_h5: null pointer");
    return B2H_EINVAL;
  }
  if (pad_mode != B2H_PAD_REPEAT_FIRST && pad_mode != B2H_PAD_ZEROS) { set_error("b2h_preprocess_h5: bad pad_mode %d", pad_mode); return B2H_EINVAL; }
  if (n_frames < 0 || n_win < 0 || T < 0) { set_error("b2h_preprocess_h5: negative size"); return B2H_ESHAPE; }
  PreArgs p{};
  p.src[0] = rows150; p.src[1] = nullptr; p.src[2] = nullptr;
  p.n_frames = n_frames; p.win_start = win_start; p.win_end = win_end; p.n_win = n_win; p.T = T; p.pad_mode = pad_mode;
  p.dif = dif_encoding; p.normalize = normalize; p.factor = factor;
  p.rfactor = 1.0f / factor; p.fastdiv = (factor == 1280.0f) ? 1 : 0;   // the reference's factor (run.py:90): verified exhaustively
  p.out[0] = input_kp; p.out[1] = input_conf; p.out[2] = target_kp; p.out[3] = target_conf;
  p.out[4] = left_kp; p.out[5] = left_conf;
  p.n_frames_out = n_frames_out; p.input_bf16 = nullptr;
  bool al = aligned16(rows150);
  for (int a = 0; a < 6; ++a) al = al && aligned16(p.out[a]);
  if (!al) { set_error("b2h_preprocess_h5: pointers must be 16-byte aligned"); return B2H_EALIGN; }
  p.aligned = 1;
  return launch_pre<1>(p, (cudaStream_t)stream);
}
