// K3: gradient-partial reduction, fused Adam (+ re-pack of the updated weights into every operand
// layout the conv kernels read), stand-alone weight packing, and the stand-alone criteria kernels of
// the modular API (mask_output, maskedPoseL1 / poderatedPoseL1 value + gradient).
//
// Reference semantics (paths relative to the reference root):
//   torch.optim.Adam(model.parameters(), lr)   body2hand/src/steps/traintest.py:48, :119-121
//   mask_output                                body2hand/src/steps/utils.py:309-312
//   maskedPoseL1 / poderatedPoseL1             body2hand/src/steps/utils.py:413-452
#include "b2h_common.cuh"

namespace b2h {

__global__ void pack_kernel(const float* __restrict__ params, char* packed, Geo g) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < g.P) scatter_packed(g, packed, gp_slot_of_flat(g, i), params[i]);
}

// Cross-CTA partial sum, shared by the reduce and the Adam kernel.  A block owns 32 consecutive slots of the
// partial layout (coalesced 128-B rows); its 8 warps each sum every 8th CTA slice, then combine through smem.
// Fixed order -> deterministic.  Returns the total in warp 0 (all lanes), garbage elsewhere.
__device__ __forceinline__ float block_partial_sum(const float* __restrict__ partials, int nparts, size_t stride, int j, int nj,
                                                   float (*red)[32]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (j < nj) {
    int c = warp;
    for (; c + 24 < nparts; c += 32) {
      s0 += partials[(size_t)c * stride + j];
      s1 += partials[(size_t)(c + 8) * stride + j];
      s2 += partials[(size_t)(c + 16) * stride + j];
      s3 += partials[(size_t)(c + 24) * stride + j];
    }
    for (; c < nparts; c += 8) s0 += partials[(size_t)c * stride + j];
  }
  red[warp][lane] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  float s = 0.f;
  if (warp == 0) {
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][lane];
  }
  return s;
}

__device__ __forceinline__ void loss_partial_sum(const float* __restrict__ loss_partials, int nparts, float* __restrict__ loss_out) {
  if (blockIdx.x == 0 && threadIdx.x < 32 && loss_out) {
    float s = 0.f;
    for (int c = threadIdx.x; c < nparts; c += 32) s += loss_partials[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) *loss_out = s;
  }
}

// grads[i] = sum_c partials[c][slot(i)];  loss = sum_c loss_partials[c]
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partials, int nparts, int gp_layout, Geo g,
                                                              float* __restrict__ grads, const float* __restrict__ loss_partials,
                                                              float* __restrict__ loss_out, const long long* __restrict__ epoch_dev,
                                                              int n_loss_parts) {
  __shared__ float red[8][32];
  if (epoch_dev) grads += (size_t)(*epoch_dev & 1) * g.P;      // data parallel: double-buffered exchange slot
  const int nj = gp_layout ? gp_total(g) : g.P;
  const int j = blockIdx.x * 32 + (threadIdx.x & 31);
  const float s = block_partial_sum(partials, nparts, (size_t)nj, j, nj, red);
  if (threadIdx.x < 32 && j < nj) {
    const int i = gp_layout ? flat_index_of_gp(g, j) : j;
    if (i >= 0) grads[i] = s;
  }
  loss_partial_sum(loss_partials, n_loss_parts, loss_out);
}

struct AdamArgs {
  float* params; const float* grads; int nparts; int gp_layout; int64_t n;
  float* m; float* v;
  float beta1, beta2, one_minus_b1, one_minus_b2, step_size, inv_bc2_sqrt, eps, grad_scale;
  double lr_d, beta1_d, beta2_d;
  long long step_host;
  const long long* step_dev;
  const double* lr_dev;            // nullable: learning rate in device memory (captured graphs follow lr changes)
  char* packed; Geo g;
  const float* loss_partials; float* loss_out; int n_loss_parts;
};

// Bias corrections step_size = lr/(1-b1^t), inv_bc2_sqrt = 1/sqrt(1-b2^t) from the device-side step counter / learning rate
// (graph replay), computed by one thread of a block.  Three forms of these coefficients exist, and each stays as it is
// because switching a path to another form moves its trained weights in the last bits:
//   - the Adam kernels of this file, when step_dev or lr_dev is given: this function, double precision with ipow;
//   - launch_adam on the host for calls without step_dev / lr_dev: double-precision pow();
//   - the fused tail of conv_tc_tile_kernel: fp32 -expm1f(t * log1pf(beta - 1)), because double-precision powers cost
//     ~5k cycles on B200's few FP64 units inside the one-launch train step.
__device__ __forceinline__ void adam_bias_corrections(const AdamArgs& a, float& step_size, float& inv_bc2_sqrt) {
  const long long t = a.step_dev ? *a.step_dev : a.step_host;
  const double lr = a.lr_dev ? *a.lr_dev : a.lr_d;
  step_size = (float)(lr / (1.0 - ipow(a.beta1_d, t)));
  inv_bc2_sqrt = (float)(1.0 / sqrt(1.0 - ipow(a.beta2_d, t)));
}

// torch.optim.Adam single-tensor update (adam_update) over the flat buffers, 32 slots per block
__global__ void __launch_bounds__(256) adam_kernel(AdamArgs a) {
  __shared__ float red[8][32];
  __shared__ float s_step_size, s_inv_bc2_sqrt;
  if (a.step_dev || a.lr_dev) {
    if (threadIdx.x == 0) adam_bias_corrections(a, s_step_size, s_inv_bc2_sqrt);
    __syncthreads();
    a.step_size = s_step_size;
    a.inv_bc2_sqrt = s_inv_bc2_sqrt;
  }
  const int nj = a.gp_layout ? gp_total(a.g) : (int)a.n;
  const int j = blockIdx.x * 32 + (threadIdx.x & 31);
  float gr;
  if (a.nparts == 1) {            // already-reduced flat gradient (modular / data-parallel path)
    gr = (j < nj && threadIdx.x < 32) ? a.grads[j] : 0.f;
  } else {
    gr = block_partial_sum(a.grads, a.nparts, (size_t)nj, j, nj, red);
  }
  if (threadIdx.x < 32 && j < nj) {
    const int i = a.gp_layout ? flat_index_of_gp(a.g, j) : j;
    if (i >= 0) {
      float m = a.m[i], v = a.v[i];
      const float p = adam_update(m, v, a.params[i], gr * a.grad_scale, a.one_minus_b1, a.one_minus_b2, a.beta2, a.eps,
                                  a.step_size, a.inv_bc2_sqrt);
      a.m[i] = m; a.v[i] = v; a.params[i] = p;
      if (a.packed) scatter_packed(a.g, a.packed, gp_slot_of_flat(a.g, i), p);
    }
  }
  loss_partial_sum(a.loss_partials, a.n_loss_parts, a.loss_out);
}

// Few gradient slices (wide training: split-K factor 6..37; small batches of the tile kernel): Adam with BOTH sides coalesced.
// The gradient slices are in slot order [k][ci/4][co][4] (what the TMEM read-out writes), the parameters / moments in the
// reference's (co, ci, k) order: one thread per slot made every m / v / p access and most packed-operand stores hit their
// own 32-byte sector (ncu at C = 256: 302 MB of DRAM writes for 3 MB of parameters, 87 us).  Here a block owns 2 output
// channels of one layer: (1) sum the slices in slot order (32-B runs) into shared memory [co][ci][k], (2) walk the flat
// order -- cin*5 contiguous floats per output channel -- for the Adam update, (3) scatter the new weights into the packed
// operand layouts in slot order, where their stores coalesce.  Fixed summation order -> deterministic.
constexpr int kAdamCoGroup = 2;   // output channels per block: 406 blocks at C = 256 (latency-bound kernel: many small blocks)
__global__ void __launch_bounds__(256) adam_gp_tile_kernel(AdamArgs a) {
  extern __shared__ float g_s[];                      // [kAdamCoGroup][kp][5] gradient sums, then the new weights
  __shared__ float s_step_size, s_inv_bc2_sqrt;
  __shared__ float b_s[kAdamCoGroup];
  const Geo& g = a.g;
  if (a.step_dev || a.lr_dev) {
    if (threadIdx.x == 0) adam_bias_corrections(a, s_step_size, s_inv_bc2_sqrt);
  } else if (threadIdx.x == 0) {
    s_step_size = a.step_size; s_inv_bc2_sqrt = a.inv_bc2_sqrt;
  }
  // block -> (layer, first output channel)
  int l = 0, b = blockIdx.x;
  for (int q = 0; q < 4; ++q) {
    const int nb = (g.cout[q] + kAdamCoGroup - 1) / kAdamCoGroup;
    if (b >= nb && q < 3) { b -= nb; l = q + 1; } else break;
  }
  const int co0 = b * kAdamCoGroup;
  const int kp = g.kp[l], cin = g.cin[l], cout = g.cout[l], q4 = kp >> 2;
  const int nj = gp_total(g);
  const size_t base = (size_t)gp_layer_off(g, l);
  const int nslot = B2H_KW * q4 * kAdamCoGroup * 4;
  // (1) slot order: idx = ((k * q4 + q) * 4 + cl) * 4 + e  ->  64-byte runs of the slices
  for (int idx = threadIdx.x; idx < nslot; idx += blockDim.x) {
    const int e = idx & 3, cl = (idx >> 2) % kAdamCoGroup, r = idx / (4 * kAdamCoGroup);
    const int q = r % q4, k = r / q4;
    const int co = co0 + cl;
    float s = 0.f;
    if (co < cout) {
      const float* src = a.grads + base + ((size_t)(k * q4 + q) * cout + co) * 4 + e;
      for (int c0 = 0; c0 < a.nparts; c0 += 8) {         // 8 independent loads in flight, summed in slice order
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (c0 + u < a.nparts) ? __ldcs(src + (size_t)(c0 + u) * nj) : 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u) s += v[u];
      }
    }
    g_s[(cl * kp + 4 * q + e) * B2H_KW + k] = s;
  }
  if (threadIdx.x < kAdamCoGroup) {
    const int co = co0 + threadIdx.x;
    float s = 0.f;
    if (co < cout) {
      const size_t j = base + (size_t)B2H_KW * cout * kp + co;
      for (int c = 0; c < a.nparts; ++c) s += __ldcs(a.grads + (size_t)c * nj + j);     // same slice order as above
    }
    b_s[threadIdx.x] = s;
  }
  __syncthreads();
  const float step_size = s_step_size, inv_bc2_sqrt = s_inv_bc2_sqrt;
  auto adam1 = [&](int i, float gr) {
    float m = a.m[i], v = a.v[i];
    const float p = adam_update(m, v, a.params[i], gr * a.grad_scale, a.one_minus_b1, a.one_minus_b2, a.beta2, a.eps, step_size,
                                inv_bc2_sqrt);
    a.m[i] = m; a.v[i] = v; a.params[i] = p;
    return p;
  };
  // (2) flat order: the cin*5 weights of one output channel are contiguous
  for (int cl = 0; cl < kAdamCoGroup; ++cl) {
    const int co = co0 + cl;
    if (co >= cout) break;
    const int i0 = g.w_off[l] + co * cin * B2H_KW;
    for (int r = threadIdx.x; r < cin * B2H_KW; r += blockDim.x) {
      const int ci = r / B2H_KW, k = r - ci * B2H_KW;
      float* gs = &g_s[(cl * kp + ci) * B2H_KW + k];
      *gs = adam1(i0 + r, *gs);
    }
  }
  if (threadIdx.x < kAdamCoGroup && co0 + (int)threadIdx.x < cout) {
    const int co = co0 + threadIdx.x;
    const float p = adam1(g.b_off[l] + co, b_s[threadIdx.x]);
    if (a.packed) scatter_packed(g, a.packed, GpSlot{l, 0, co, 0, true}, p);
  }
  __syncthreads();
  // (3) slot order again: scatter the new weights into the packed operand layouts
  if (a.packed) {
    for (int idx = threadIdx.x; idx < nslot; idx += blockDim.x) {
      const int e = idx & 3, cl = (idx >> 2) % kAdamCoGroup, r = idx / (4 * kAdamCoGroup);
      const int q = r % q4, k = r / q4;
      const int co = co0 + cl, ci = 4 * q + e;
      if (co < cout && ci < cin) scatter_packed(g, a.packed, GpSlot{l, k, co, ci, false}, g_s[(cl * kp + ci) * B2H_KW + k]);
    }
  }
  loss_partial_sum(a.loss_partials, a.n_loss_parts, a.loss_out);
}

// Few slices, small model (conv_channels ~ 64): one thread per gradient-partial slot, coalesced loads of the slot from every
// slice (fixed order -> deterministic), Adam, scatter into the packed operand layouts.  (adam_kernel's 32-slots-per-block
// shape is built for ~20k slots x 128 slices; adam_gp_tile_kernel needs >= ~100 blocks of work to fill the chip.)
__global__ void __launch_bounds__(256) adam_gp_wide_kernel(AdamArgs a) {
  __shared__ float s_step_size, s_inv_bc2_sqrt;
  if (a.step_dev || a.lr_dev) {
    if (threadIdx.x == 0) adam_bias_corrections(a, s_step_size, s_inv_bc2_sqrt);
    __syncthreads();
    a.step_size = s_step_size;
    a.inv_bc2_sqrt = s_inv_bc2_sqrt;
  }
  const int nj = gp_total(a.g);
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < nj) {
    float gr = 0.f;
    for (int c = 0; c < a.nparts; ++c) gr += __ldcs(a.grads + (size_t)c * nj + j);
    GpSlot sl;
    if (gp_decode(a.g, j, sl)) {
      const int i = gp_flat_of_slot(a.g, sl);
      float m = a.m[i], v = a.v[i];
      const float p = adam_update(m, v, a.params[i], gr * a.grad_scale, a.one_minus_b1, a.one_minus_b2, a.beta2, a.eps,
                                  a.step_size, a.inv_bc2_sqrt);
      a.m[i] = m; a.v[i] = v; a.params[i] = p;
      if (a.packed) scatter_packed(a.g, a.packed, sl, p);
    }
  }
  loss_partial_sum(a.loss_partials, a.n_loss_parts, a.loss_out);
}

// grads[i] = sum_c partials[c][slot(i)] for the same shape of problem (one thread per slot)
__global__ void __launch_bounds__(256) reduce_gp_wide_kernel(const float* __restrict__ partials, int nparts, Geo g, float* __restrict__ grads,
                                                             const float* __restrict__ loss_partials, float* __restrict__ loss_out,
                                                             const long long* __restrict__ epoch_dev, int n_loss_parts) {
  if (epoch_dev) grads += (size_t)(*epoch_dev & 1) * g.P;
  const int nj = gp_total(g);
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < nj) {
    float s = 0.f;
    for (int c = 0; c < nparts; ++c) s += __ldcs(partials + (size_t)c * nj + j);
    const int i = flat_index_of_gp(g, j);
    if (i >= 0) grads[i] = s;
  }
  loss_partial_sum(loss_partials, n_loss_parts, loss_out);
}

// ---- data parallel: gradient exchange over peer (NVLink) memory fused with Adam -------------------------------
// Three-launch path of b2h_train_step_dp (shapes the one-launch tile kernel does not serve): train kernel, reduce_* into
// this rank's buffer, adam_dp_kernel.
// Every rank owns a symmetric buffer  [2][P] fp32 gradients (double-buffered by epoch parity) + [world] int64 flags.
// Step protocol (one kernel per rank, all ranks run it concurrently on their own GPU):
//   1. block 0 publishes "my gradients of epoch e are complete" by storing e into flag[rank] of every peer
//      (the reduce kernel that wrote them is the previous kernel on the stream; __threadfence_system orders it);
//   2. every block waits until all world flags in the LOCAL buffer have reached e (acquire loads, bounded spin);
//   3. every thread sums its gradient element over the peers' buffers in rank order (identical arithmetic on
//      every rank -> replicas stay bit-identical) and applies Adam + weight re-pack.
// Re-use safety: a rank can be at most one epoch ahead of a peer (it needs the peer's flag for e+1 to pass 2.),
// and epoch e+1 uses the other half of the buffer, so nobody overwrites data that is still being read.
__device__ int g_dp_status = 0;

struct AdamDpArgs {
  AdamArgs a;
  const float* const* peer_bufs;   // device array [world] of peer buffer base pointers (index = rank)
  const long long* epoch_dev;
  int rank, world;
};

__global__ void __launch_bounds__(256) adam_dp_kernel(AdamDpArgs d) {
  AdamArgs& a = d.a;
  __shared__ float s_step_size, s_inv_bc2_sqrt;
  const long long epoch = *d.epoch_dev;
  const size_t P = (size_t)a.n;
  const size_t flag_off = 2 * P;                       // in floats; flags are 8-byte aligned (2P is even)
  __shared__ int s_abort;
  if (threadIdx.x == 0) {
    adam_bias_corrections(a, s_step_size, s_inv_bc2_sqrt);
    s_abort = 0;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x < d.world) {
    __threadfence_system();
    volatile long long* f = reinterpret_cast<volatile long long*>(const_cast<float*>(d.peer_bufs[threadIdx.x]) + flag_off) + d.rank;
    *f = epoch;
    __threadfence_system();
  }
  if (threadIdx.x < d.world) {
    const volatile long long* f = reinterpret_cast<const volatile long long*>(d.peer_bufs[d.rank] + flag_off) + threadIdx.x;
    const long long t0 = clock64();
    while (*f < epoch) {
      if (clock64() - t0 > 6000000000LL) { atomicExch(&g_dp_status, 1); s_abort = 1; break; }   // ~3 s: never hang the box
    }
    __threadfence_system();
  }
  __syncthreads();
  // Sticky abort: once a peer wait has timed out, no parameter / moment is written (this step and every later one)
  // until the host has read and cleared the status -- replicas may stall, they never silently diverge.
  if (s_abort || *reinterpret_cast<volatile int*>(&g_dp_status) != 0) return;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < a.n) {
    const size_t off = (size_t)(epoch & 1) * P + (size_t)i;
    float gr = 0.f;
    for (int r = 0; r < d.world; ++r) gr += __ldcv(d.peer_bufs[r] + off);
    float m = a.m[i], v = a.v[i];
    const float p = adam_update(m, v, a.params[i], gr * a.grad_scale, a.one_minus_b1, a.one_minus_b2, a.beta2, a.eps, s_step_size,
                                s_inv_bc2_sqrt);
    a.m[i] = m; a.v[i] = v; a.params[i] = p;
    if (a.packed) scatter_packed(a.g, a.packed, gp_slot_of_flat(a.g, (int)i), p);
  }
}

// The AdamArgs fields every Adam launch sets the same way; the caller adds where the gradients come from and the host-side
// bias corrections.
static AdamArgs adam_args(float* params, float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps,
                          long long step, const long long* step_dev, const double* lr_dev, float grad_scale, void* packed,
                          const Geo& g) {
  AdamArgs a{};
  a.params = params; a.n = n; a.m = m; a.v = v;
  a.beta1 = (float)beta1; a.beta2 = (float)beta2;
  a.one_minus_b1 = (float)(1.0 - beta1); a.one_minus_b2 = (float)(1.0 - beta2);
  a.eps = (float)eps; a.grad_scale = grad_scale;
  a.packed = reinterpret_cast<char*>(packed); a.g = g;
  a.lr_d = lr; a.beta1_d = beta1; a.beta2_d = beta2; a.step_dev = step_dev; a.lr_dev = lr_dev; a.step_host = step;
  return a;
}

int launch_adam_dp(float* params, const float* const* peer_bufs, int rank, int world, float* m, float* v, int64_t n, double lr,
                   double beta1, double beta2, double eps, const long long* step_dev, const long long* epoch_dev, const double* lr_dev,
                   float grad_scale, void* packed, const Geo& g, cudaStream_t stream) {
  AdamDpArgs d{};
  d.a = adam_args(params, m, v, n, lr, beta1, beta2, eps, 1, step_dev, lr_dev, grad_scale, packed, g);
  d.peer_bufs = peer_bufs; d.epoch_dev = epoch_dev; d.rank = rank; d.world = world;
  adam_dp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(d);
  count_launch();
  return check_launch("adam_dp_kernel");
}

int dp_status_and_clear() {
  int v = 0, z = 0;
  cudaMemcpyFromSymbol(&v, g_dp_status, sizeof(int));
  if (v) cudaMemcpyToSymbol(g_dp_status, &z, sizeof(int));
  return v;
}

__global__ void mask_output_kernel(float* __restrict__ y, const int32_t* __restrict__ lengths, int B, int T, int row) {
  const int64_t n = (int64_t)B * T * row;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bt = i / row;
    const int b = (int)(bt / T), t = (int)(bt - (int64_t)b * T);
    if (t >= lengths[b]) y[i] = 0.0f;                     // output[i, len:, :] = 0   utils.py:311
  }
}

// one CTA per sample: per-sample mean |d| over the first len frames (+ gradient)
__global__ void __launch_bounds__(256) pose_l1_rows_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                           const float* __restrict__ scores,
                                                           const int32_t* __restrict__ lengths, int B, int T, int row,
                                                           int loss_kind, float* __restrict__ d_pred,
                                                           float* __restrict__ row_scratch) {
  __shared__ float red[8];
  const int b = blockIdx.x;
  int len = lengths[b];
  len = len < 0 ? 0 : (len > T ? T : len);
  const float n_el = (float)len * (float)row;
  const float scale = (loss_kind == B2H_LOSS_L1) ? (1.0f / (float)B) / n_el : 1.0f / n_el;
  const size_t base = (size_t)b * T * row;
  float sum = 0.f;
  for (int i = threadIdx.x; i < T * row; i += blockDim.x) {
    const int t = i / row;
    float gr = 0.f;
    if (t < len) {
      const float pr = pred[base + i], tv = target[base + i];
      float d, s = 1.f;
      if (loss_kind == B2H_LOSS_L1) {
        d = pr - tv;
      } else {
        s = scores[((size_t)b * T + t) * (row >> 1) + ((i - t * row) >> 1)];
        d = __fsub_rn(__fmul_rn(pr, s), __fmul_rn(tv, s));
      }
      sum += fabsf(d);
      gr = (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) * s * scale;
    }
    if (d_pred) d_pred[base + i] = gr;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    row_scratch[b] = s / n_el;
  }
}

__global__ void pose_l1_final_kernel(const float* __restrict__ row_scratch, int B, int loss_kind, float* __restrict__ loss_out) {
  // sequential like the reference's python loop (loss += ...), then / B for maskedPoseL1
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += row_scratch[b];
    *loss_out = (loss_kind == B2H_LOSS_L1) ? s / (float)B : s;
  }
}

// Inference output formats (SURVEY 8f N2).  pred (R,42) = rows of [x0,y0,x1,y1,...] ->
//   mode 0: OpenPose hand rows [x0,y0,1.0, x1,y1,1.0, ...] (63)      array2open_pose        steps/utils.py:355-364
//   mode 1: packed H5 rows     [x0..x20 | y0..y20 | 0 x 21]  (63)      order_and_reshape_toh5 steps/traintest.py:302-317
__global__ void format_prediction_kernel(const float* __restrict__ pred, float* __restrict__ out, int64_t rows, int mode) {
  const int64_t n = rows * 63;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / 63;
    const int c = (int)(i - r * 63);
    float v;
    if (mode == 0) {
      const int j = c / 3, d = c - j * 3;
      v = d == 2 ? 1.0f : pred[r * 42 + 2 * j + d];
    } else {
      const int d = c / 21, j = c - d * 21;
      v = d == 2 ? 0.0f : pred[r * 42 + 2 * j + d];
    }
    out[i] = v;
  }
}

// LinearPositionalEmbedding.forward  body2hand/src/models/HandPoseModels.py:78-84: out (B, C+1, T) = cat([t / max_len, inp (B, C, T)], dim=1)
__global__ void pos_emb_concat_kernel(const float* __restrict__ inp, float* __restrict__ out, int B, int Cc, int T, float max_len) {
  const int64_t n = (int64_t)B * (Cc + 1) * T;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int t = (int)(i % T);
    const int64_t bc = i / T;
    const int c = (int)(bc % (Cc + 1));
    const int64_t b = bc / (Cc + 1);
    out[i] = c == 0 ? __fdiv_rn((float)t, max_len) : inp[(b * Cc + (c - 1)) * T + t];
  }
}

int launch_pos_emb_concat(const float* inp, float* out, int B, int Cc, int T, int max_len, cudaStream_t stream) {
  const int64_t n = (int64_t)B * (Cc + 1) * T;
  if (n == 0) return B2H_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  pos_emb_concat_kernel<<<(unsigned)blocks, 256, 0, stream>>>(inp, out, B, Cc, T, (float)max_len);
  count_launch();
  return check_launch("pos_emb_concat_kernel");
}

int launch_format_prediction(const float* pred, float* out, int64_t rows, int mode, cudaStream_t stream) {
  if (rows == 0) return B2H_OK;
  int64_t blocks = (rows * 63 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  format_prediction_kernel<<<(unsigned)blocks, 256, 0, stream>>>(pred, out, rows, mode);
  count_launch();
  return check_launch("format_prediction_kernel");
}

int launch_pack(const float* params, void* packed, const Geo& g, cudaStream_t stream) {
  pack_kernel<<<(g.P + 255) / 256, 256, 0, stream>>>(params, reinterpret_cast<char*>(packed), g);
  count_launch();
  return check_launch("pack_kernel");
}

// Few gradient slices in the slot layout (wide training, small batches of the tile kernel): the reduction and Adam kernels
// that sum every slice of a slot in one thread, instead of spreading the slices over the 8 warps of a block.
static bool few_slices(int nparts, int gp_layout) { return gp_layout && nparts <= 64; }

int launch_reduce(const float* partials, int nparts, int gp_layout, const Geo& g, float* grads, const float* loss_partials,
                  float* loss_out, cudaStream_t stream, const long long* epoch_dev, int n_loss_parts) {
  const int nj = gp_layout ? gp_total(g) : g.P;
  if (few_slices(nparts, gp_layout)) {                 // one thread per slot
    reduce_gp_wide_kernel<<<(nj + 255) / 256, 256, 0, stream>>>(partials, nparts, g, grads, loss_partials, loss_out, epoch_dev,
                                                                n_loss_parts < 0 ? nparts : n_loss_parts);
    count_launch();
    return check_launch("reduce_gp_wide_kernel");
  }
  reduce_partials_kernel<<<(nj + 31) / 32, 256, 0, stream>>>(partials, nparts, gp_layout, g, grads, loss_partials, loss_out, epoch_dev,
                                                             n_loss_parts < 0 ? nparts : n_loss_parts);
  count_launch();
  return check_launch("reduce_partials_kernel");
}

int launch_adam(float* params, const float* grads, int nparts, int gp_layout, float* m, float* v, int64_t n, double lr, double beta1,
                double beta2, double eps, int64_t step, const long long* step_dev, const double* lr_dev, float grad_scale, void* packed,
                const Geo& g, const float* loss_partials, float* loss_out, cudaStream_t stream, int n_loss_parts) {
  AdamArgs a = adam_args(params, m, v, n, lr, beta1, beta2, eps, step, step_dev, lr_dev, grad_scale, packed, g);
  a.grads = grads; a.nparts = nparts; a.gp_layout = gp_layout;
  a.loss_partials = loss_partials; a.loss_out = loss_out; a.n_loss_parts = n_loss_parts < 0 ? nparts : n_loss_parts;
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  a.step_size = (float)(lr / bc1);
  a.inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
  const int64_t nj = gp_layout ? (int64_t)gp_total(g) : n;
  if (few_slices(nparts, gp_layout) && nj <= 100000) { // small model: one thread per slot
    adam_gp_wide_kernel<<<(unsigned)((nj + 255) / 256), 256, 0, stream>>>(a);
    count_launch();
    return check_launch("adam_gp_wide_kernel");
  }
  if (few_slices(nparts, gp_layout)) {                 // large model (wide training): coalesced on both sides
    int blocks = 0, kpmax = 0;
    for (int l = 0; l < 4; ++l) { blocks += (g.cout[l] + kAdamCoGroup - 1) / kAdamCoGroup; kpmax = g.kp[l] > kpmax ? g.kp[l] : kpmax; }
    const size_t smem = (size_t)kAdamCoGroup * kpmax * B2H_KW * sizeof(float);
    adam_gp_tile_kernel<<<blocks, 256, smem, stream>>>(a);
    count_launch();
    return check_launch("adam_gp_tile_kernel");
  }
  if (nparts == 1) adam_kernel<<<(unsigned)((nj + 31) / 32), 32, 0, stream>>>(a);
  else adam_kernel<<<(unsigned)((nj + 31) / 32), 256, 0, stream>>>(a);
  count_launch();
  return check_launch("adam_kernel");
}

int launch_mask_output(float* y, const int32_t* lengths, int B, int T, int row, cudaStream_t stream) {
  int64_t n = (int64_t)B * T * row;
  if (n == 0) return B2H_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  mask_output_kernel<<<(unsigned)blocks, 256, 0, stream>>>(y, lengths, B, T, row);
  count_launch();
  return check_launch("mask_output_kernel");
}

int launch_pose_l1(const float* pred, const float* target, const float* scores, const int32_t* lengths, int B, int T,
                   int row, int loss_kind, float* loss_out, float* d_pred, float* row_scratch, cudaStream_t stream) {
  if (B <= 0) return B2H_OK;
  pose_l1_rows_kernel<<<B, 256, 0, stream>>>(pred, target, scores, lengths, B, T, row, loss_kind, d_pred, row_scratch);
  pose_l1_final_kernel<<<1, 32, 0, stream>>>(row_scratch, B, loss_kind, loss_out);
  count_launch(2);
  return check_launch("pose_l1 kernels");
}

}  // namespace b2h
