// Forward, training and validation over packed utterances and segments (b2h_conv_forward_utterances,
// b2h_train_*_utterances, b2h_validate_utterances): the device-side plan and the one launcher.  Included by b2h_conv_tc.cu
// after the tile and wide kernels.
//
// Utterance u owns stream rows [offsets[u], offsets[u+1]) and is predicted as ONE sequence, like the reference's
// infer_utterance (steps/traintest.py:214-300): it is cut into sub-windows of Ts frames by the training cut rule
// (sub_window(), b2h_common.cuh), every interior cut with >= 16 real frames of context on both sides.  The receptive field
// of the four convolutions is +-8 frames, so a sub-window's core rows equal the whole sequence's rows there; the utterance
// start is the window's own leading zero rows, and rows at or past the utterance end are zero in every layer.
//
// The offsets live on the device, so the host sizes the launch from a bound (UttPlan::max_sub) and a one-CTA planning
// kernel turns the offsets into the sub-window table the forward kernels read (layout: UttPlan).  The forward kernels end
// their tile loops at the table's count.
//
// Training over segments (b2h_train_*_utterances) plans the same way: segment s = stream rows [seg_start[s], seg_end[s]),
// 1..max_len frames, trained as one sequence; the planning kernel also writes each sub-window's segment and its length
// (loss weight 1 / (42 L_s)) and the "bad" word the fused step reads before its Adam update.
#pragma once

namespace b2h {

constexpr int kUttPlanThreads = 1024;
constexpr int kUttBadOffsets = 80;   // b2h_tc_status id: offsets not non-decreasing within [0, n_frames]
constexpr int kUttBadSegments = 81;  // b2h_tc_status id: a training segment outside [0, n_frames] or not of 1..max_len frames

// Sequence u is rows [seg_a[u], seg_b[u]): the offsets form of the forward passes (off, off + 1).  max_len > 0 (training):
// every sequence must hold 1..max_len frames, and seg_out receives {u, L_u} per sub-window.
__global__ void __launch_bounds__(kUttPlanThreads) utt_plan_kernel(const long long* __restrict__ seg_a, const long long* __restrict__ seg_b,
                                                                   int n_utt, long long n_frames, int Ts, int max_sub, int max_len,
                                                                   int bad_id, int4* ws, int2* seg_out) {
  __shared__ int warp_sum[32];
  __shared__ int s_bad;
  int4* table = ws + 1;
  int* prefix = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + utt_prefix_offset(max_sub));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  griddep_launch_dependents();       // the forward behind it may start its set-up; it reads the table after griddep_wait
  if (tid == 0) s_bad = 0;
  __syncthreads();
  // pass 1: check the offsets, count each utterance's sub-windows, exclusive prefix sum (1024 utterances per round)
  long long carry = 0;
  for (int base = 0; base < n_utt; base += kUttPlanThreads) {
    const int u = base + tid;
    int cnt = 0;
    if (u < n_utt) {
      const long long a = seg_a[u], b = seg_b[u];
      if (a < 0 || b < a || b > n_frames || (max_len > 0 && (b == a || b - a > max_len))) s_bad = 1;
      else cnt = sub_window_count(b - a, Ts);
    }
    int v = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += n;
    }
    if (lane == 31) warp_sum[warp] = v;
    __syncthreads();
    if (warp == 0) {
      int w = warp_sum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += n;
      }
      warp_sum[lane] = w;
    }
    __syncthreads();
    const long long excl = carry + (v - cnt) + (warp ? warp_sum[warp - 1] : 0);
    if (u < n_utt) prefix[u] = excl < max_sub ? (int)excl : max_sub;
    carry += warp_sum[31];
    __syncthreads();
  }
  // valid offsets hold at most n_frames frames, so carry <= max_sub (sub_window_count); bad ones plan nothing
  const bool bad = s_bad || carry > max_sub;
  const int count = bad ? 0 : (int)carry;
  if (tid == 0) {
    prefix[n_utt] = count;
    ws[0] = make_int4(count, bad ? 1 : 0, 0, 0);
    if (bad) atomicExch(&g_tc_status, bad_id);
  }
  __syncthreads();                   // the prefix sums are visible to the whole CTA
  // pass 2: sub-window g -> (utterance u, index i) by binary search over the prefix sums -> sub_window()
  for (int gi = tid; gi < count; gi += kUttPlanThreads) {
    int lo = 0, hi = n_utt - 1;      // the last u with prefix[u] <= gi (empty utterances share their successor's prefix)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (prefix[mid] <= gi) lo = mid;
      else hi = mid - 1;
    }
    const int n = prefix[lo + 1] - prefix[lo], i = gi - prefix[lo];
    const long long a = seg_a[lo];
    const int L = (int)(seg_b[lo] - a);
    int start = 0, clo = 0, chi = L;
    if (n > 1) {
      const SubWindow s = sub_window(L, Ts, n, i);
      start = s.start; clo = s.clo; chi = s.chi;
    }
    const int len = L - start < Ts ? L - start : Ts;
    table[gi] = make_int4((int)(a + start), start, clo | (chi << 16), len);
    if (seg_out) seg_out[gi] = make_int2(lo, L);
  }
}

// Validation over segments, the last launch: seg_loss[s] = (the sums of segment s's sub-windows, in table order) / (42 L_s);
// loss = the sum over s in a fixed order (per-thread strided sums, then a fixed tree), times 1 / S for L1.  A refused plan:
// NaN in loss and every seg_loss entry.
__global__ void __launch_bounds__(kUttPlanThreads) utt_validate_finish_kernel(const int4* __restrict__ ws, const int2* __restrict__ seg,
                                                                              const float* __restrict__ part, int n_seg, int max_sub,
                                                                              int loss_kind, float* seg_loss, float* loss_out) {
  __shared__ float warp_sum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  griddep_wait();                    // the forward's sums are complete and visible
  const bool bad = __ldg(&ws->y) != 0;
  const int* prefix = reinterpret_cast<const int*>(reinterpret_cast<const char*>(ws) + utt_prefix_offset(max_sub));
  const float nan = __int_as_float(0x7fffffff);
  float acc = 0.f;
  for (int s = tid; s < n_seg; s += kUttPlanThreads) {
    float v = nan;
    if (!bad) {
      const int g0 = __ldg(prefix + s), g1 = __ldg(prefix + s + 1);
      float sum = 0.f;
      for (int gi = g0; gi < g1; ++gi) sum += __ldg(part + gi);
      v = sum / ((float)__ldg(&seg[g0].y) * (float)B2H_COUT);   // every segment has >= 1 sub-window: seg[g0] is its own
      acc += v;
    }
    if (seg_loss) seg_loss[s] = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) warp_sum[warp] = acc;
  __syncthreads();
  if (tid == 0) {
    float total = 0.f;
    for (int w = 0; w < kUttPlanThreads / 32; ++w) total += warp_sum[w];
    *loss_out = bad ? nan : (loss_kind == B2H_LOSS_L1 ? total / (float)n_seg : total);
  }
}

int launch_utterances(ConvArgs a, const UttPlan& plan, const SegmentView& sv, void* table, float* seg_loss, float* loss_out,
                      cudaStream_t stream) {
  int4* ws = reinterpret_cast<int4*>(table);
  int2* seg = sv.max_len > 0 ? reinterpret_cast<int2*>(reinterpret_cast<char*>(table) + plan.seg_off) : nullptr;
  utt_plan_kernel<<<1, kUttPlanThreads, 0, stream>>>(sv.seg_a, sv.seg_b, sv.n, sv.n_frames, plan.Ts, plan.max_sub, sv.max_len,
                                                     sv.max_len > 0 ? kUttBadSegments : kUttBadOffsets, ws, seg);
  count_launch();
  if (int rc = check_launch("utt_plan_kernel")) return rc;
  a.utt = ws; a.T = plan.Ts; a.lengths = nullptr;
  if (a.mode == 1) {
    a.utt_seg = seg; a.utt_max_len = sv.max_len;
    a.B = sv.n; a.apply_mask = 1;
    return launch_tc_tile(a, plan.tile, stream);
  }
  a.B = plan.max_sub; a.apply_mask = 0;
  const int rc = plan.kernel == B2H_KERNEL_TC_TILE ? launch_tc_tile(a, plan.tile, stream) : launch_tc_wide_fwd(a, plan.wide, stream);
  if (rc || !a.loss_partials) return rc;
  // validation: programmatic dependent launch, its set-up overlaps the forward's tail; it reads the sums after
  // griddepcontrol.wait
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(1); cfg.blockDim = dim3(kUttPlanThreads); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
  cudaLaunchAttribute at;
  at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &at; cfg.numAttrs = 1;
  const int4* cws = ws;
  const int2* cseg = seg;
  const float* cpart = a.loss_partials;
  int n_seg = sv.n, lk = a.loss_kind, ms = plan.max_sub;
  void* kargs[] = {&cws, &cseg, &cpart, &n_seg, &ms, &lk, &seg_loss, &loss_out};
  const cudaError_t le = cudaLaunchKernelExC(&cfg, (const void*)utt_validate_finish_kernel, kargs);
  if (le != cudaSuccess) { cudaGetLastError(); set_error("utt_validate_finish_kernel launch: %s", cudaGetErrorString(le)); return B2H_ECUDA; }
  count_launch();
  return check_launch("utt_validate_finish_kernel");
}

}  // namespace b2h
