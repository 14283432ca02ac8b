// fp32 mode (B2H_FP32): the whole ConvModel forward -- and for training the masked-L1 loss, its
// gradient and the full backward -- for one window per CTA pass, activations resident in shared
// memory, FFMA with fp32 accumulation (parity target 1e-4 relative; plain TF32 would be ~1e-3).
//
// Reference semantics (paths relative to the reference root):
//   ConvModel.forward                 body2hand/src/models/HandPoseModels.py:40-64
//   LinearPositionalEmbedding         body2hand/src/models/HandPoseModels.py:66-84
//   mask_output                       body2hand/src/steps/utils.py:309-312
//   maskedPoseL1 / poderatedPoseL1    body2hand/src/steps/utils.py:413-452
//   loss.backward()                   body2hand/src/steps/traintest.py:120 (autograd: conv dgrad /
//                                     wgrad / bias-grad, ReLU mask, L1 sign)
//
// Layout: a window's activations live in smem as rows [t+2][channel] with two zero rows in front
// and behind (the conv's zero padding), so tap k of output frame t reads row t+k.  lane -> output
// channel (coalesced tap-major weights Wf[k][ci][co] through the read-only path, conflict-free smem
// writes), each warp register-blocks 8 frames.  Gradients: every CTA owns one slice of the
// partials workspace (no atomics, deterministic); b2h_optim.cu reduces the slices.
#include "b2h_common.cuh"

namespace b2h {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;



// EPI 0: +bias, ReLU -> smem | 1: +bias -> smem | 2: no bias, multiply by (act > 0) -> smem
template <int EPI>
__device__ __forceinline__ void conv_rows(const float* __restrict__ in, int ldi, int Cin, const float* __restrict__ W,
                                          int Cout, const float* __restrict__ bias, float* __restrict__ out, int ldo,
                                          const float* __restrict__ act, int lda, int T) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nRB = (T + 7) >> 3, nCG = (Cout + 31) >> 5;
  for (int task = warp; task < nRB * nCG; task += kWarps) {
    const int rb = task / nCG, cg = task - rb * nCG;
    const int co = cg * 32 + lane;
    const bool active = co < Cout;
    const int r0 = rb * 8;
    float acc[8];
    const float b0 = (EPI != 2 && active) ? __ldg(bias + co) : 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = b0;
    const float* xin = in + r0 * ldi;
    const float* wp = W + (active ? co : 0);
    for (int ci = 0; ci < Cin; ++ci) {
      float xv[12];
#pragma unroll
      for (int j = 0; j < 12; ++j) xv[j] = xin[j * ldi + ci];
#pragma unroll
      for (int k = 0; k < B2H_KW; ++k) {
        float w = __ldg(wp + (k * Cin + ci) * Cout);
        w = active ? w : 0.0f;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv[j + k], w, acc[j]);
      }
    }
    if (active) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int t = r0 + j;
        if (t < T) {
          float v = acc[j];
          if (EPI == 0) v = fmaxf(v, 0.0f);
          if (EPI == 2) v = (act[(t + 2) * lda + co] > 0.0f) ? v : 0.0f;
          out[(t + 2) * ldo + co] = v;
        }
      }
    }
  }
}

// dW[co][ci][k] (+)= sum_t g[t][co] * a[t+k-2][ci];  db[co] (+)= sum_t g[t][co]
__device__ __forceinline__ void wgrad_rows(const float* __restrict__ g, int ldg, int Cout, const float* __restrict__ a,
                                           int lda, int Cin, float* __restrict__ pW, float* __restrict__ pB, int T,
                                           bool first) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nCG = (Cout + 31) >> 5;
  const int ntask = (Cin + 1) * nCG;          // the extra "ci" row is the bias gradient
  for (int task = warp; task < ntask; task += kWarps) {
    const int ci = task / nCG, cg = task - ci * nCG;
    const int co = cg * 32 + lane;
    const bool active = co < Cout;
    const float* gp = g + 2 * ldg + (active ? co : 0);
    if (ci < Cin) {
      float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      const float* ap = a + ci;
      float a0 = ap[0], a1 = ap[lda], a2 = ap[2 * lda], a3 = ap[3 * lda];
      for (int t = 0; t < T; ++t) {
        const float a4 = ap[(t + 4) * lda];
        const float gv = gp[t * ldg];
        acc[0] = fmaf(gv, a0, acc[0]);
        acc[1] = fmaf(gv, a1, acc[1]);
        acc[2] = fmaf(gv, a2, acc[2]);
        acc[3] = fmaf(gv, a3, acc[3]);
        acc[4] = fmaf(gv, a4, acc[4]);
        a0 = a1; a1 = a2; a2 = a3; a3 = a4;
      }
      if (active) {
        float* dst = pW + ((size_t)co * Cin + ci) * B2H_KW;
#pragma unroll
        for (int k = 0; k < B2H_KW; ++k) dst[k] = first ? acc[k] : dst[k] + acc[k];
      }
    } else {
      float s = 0.f;
      for (int t = 0; t < T; ++t) s += gp[t * ldg];
      if (active) pB[co] = first ? s : pB[co] + s;
    }
  }
}

__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) s += red[w];
  return s;
}

template <bool TRAIN>
__global__ void __launch_bounds__(kThreads) conv_fp32_kernel(ConvArgs p) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float red[kWarps];
  const Geo& g = p.geo;
  const int T = p.T;
  const int TR = round_up(T, 8) + 4;
  const int ld0 = round_up(g.cin[0], 4), ldc = round_up(g.C, 4), ldg = round_up(g.C > B2H_COUT ? g.C : B2H_COUT, 4);
  float* X = smem;
  float* A1 = X + TR * ld0;
  float* A2 = A1 + TR * ldc;
  float* A3 = A2 + TR * ldc;                      // train only
  float* G0 = A3 + TR * ldc;                      // train only
  float* G1 = G0 + TR * ldg;                      // train only
  const int total = TRAIN ? TR * (ld0 + 3 * ldc + 2 * ldg) : TR * (ld0 + 2 * ldc);
  for (int i = threadIdx.x; i < total; i += kThreads) smem[i] = 0.0f;   // zero pads once; never overwritten
  __syncthreads();

  const float* Wf[4];
  const float* Wd[4];
  const float* bias[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    Wf[l] = reinterpret_cast<const float*>(p.packed + g.wf_off[l]);
    Wd[l] = reinterpret_cast<const float*>(p.packed + g.wd_off[l]);
    bias[l] = p.params + g.b_off[l];
  }
  if (TRAIN && p.step_dev && blockIdx.x == 0 && threadIdx.x == 0) *p.step_dev += 1;
  if (TRAIN && p.epoch_dev && blockIdx.x == 0 && threadIdx.x == 0) *p.epoch_dev += 1;
  float* part = TRAIN ? p.partials + (size_t)blockIdx.x * g.P : nullptr;
  float loss_acc = 0.0f;
  bool first = true;

  for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
    // ---- stage the window: (T, n_in) NWC -> rows t+2, channel pos_emb + c ----
    const int n_in = g.n_in, pe = g.pos_emb;
    if (p.x_dtype == B2H_DT_F32) {
      const float* xs = reinterpret_cast<const float*>(p.x) + (size_t)b * T * n_in;
      for (int i = threadIdx.x; i < T * n_in; i += kThreads) {
        int t = i / n_in, c = i - t * n_in;
        X[(t + 2) * ld0 + pe + c] = __ldg(xs + i);
      }
    } else {
      const __nv_bfloat16* xs = reinterpret_cast<const __nv_bfloat16*>(p.x) + (size_t)b * T * n_in;
      for (int i = threadIdx.x; i < T * n_in; i += kThreads) {
        int t = i / n_in, c = i - t * n_in;
        X[(t + 2) * ld0 + pe + c] = __bfloat162float(xs[i]);
      }
    }
    if (pe) {   // LinearPositionalEmbedding: channel 0 = t / 100 (fp32 divide)   HandPoseModels.py:70-82
      for (int t = threadIdx.x; t < T; t += kThreads) X[(t + 2) * ld0] = __fdiv_rn((float)t, (float)g.pe_len);
    }
    __syncthreads();
    conv_rows<0>(X, ld0, g.cin[0], Wf[0], g.cout[0], bias[0], A1, ldc, nullptr, 0, T);   // HandPoseModels.py:55
    __syncthreads();
    conv_rows<0>(A1, ldc, g.cin[1], Wf[1], g.cout[1], bias[1], A2, ldc, nullptr, 0, T);  // :56
    __syncthreads();
    int len = T;
    if (p.lengths) { len = p.lengths[b]; len = len < 0 ? 0 : (len > T ? T : len); }

    if (!TRAIN) {
      conv_rows<0>(A2, ldc, g.cin[2], Wf[2], g.cout[2], bias[2], A1, ldc, nullptr, 0, T);   // :57
      __syncthreads();
      // conv4 straight to global: lane -> output channel, rows coalesced (42 floats)         :58-62
      {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int Cin = g.cin[3];
        const int nRB = (T + 7) >> 3;
        float* ys = p.y + (size_t)b * T * B2H_COUT;
        for (int task = warp; task < nRB * 2; task += kWarps) {
          const int rb = task >> 1, cg = task & 1;
          const int co = cg * 32 + lane;
          const bool active = co < B2H_COUT;
          const int r0 = rb * 8;
          float acc[8];
          const float b0 = active ? __ldg(bias[3] + co) : 0.f;
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = b0;
          const float* xin = A1 + r0 * ldc;
          const float* wp = Wf[3] + (active ? co : 0);
          for (int ci = 0; ci < Cin; ++ci) {
            float xv[12];
#pragma unroll
            for (int j = 0; j < 12; ++j) xv[j] = xin[j * ldc + ci];
#pragma unroll
            for (int k = 0; k < B2H_KW; ++k) {
              float w = __ldg(wp + (k * Cin + ci) * B2H_COUT);
              w = active ? w : 0.f;
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv[j + k], w, acc[j]);
            }
          }
          if (active) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int t = r0 + j;
              if (t < T) {
                float v = acc[j];
                if (p.apply_mask && t >= len) v = 0.0f;          // mask_output  utils.py:309-312
                else if (p.out_scale != 1.0f) v = v * p.out_scale; // prediction *= 1280  traintest.py:270-271
                ys[(size_t)t * B2H_COUT + co] = v;
              }
            }
          }
        }
      }
      __syncthreads();
      continue;
    }

    // ------------------------------ training path ------------------------------
    conv_rows<0>(A2, ldc, g.cin[2], Wf[2], g.cout[2], bias[2], A3, ldc, nullptr, 0, T);   // :57
    __syncthreads();
    if (p.mode == 1) {
      conv_rows<1>(A3, ldc, g.cin[3], Wf[3], g.cout[3], bias[3], G0, ldg, nullptr, 0, T); // :58  pred -> G0
      __syncthreads();
      // mask_output + criterion + d(loss)/d(pred), in place in G0
      const float n_el = (float)len * (float)B2H_COUT;
      const float scale = (p.loss_kind == B2H_LOSS_L1) ? (1.0f / (float)p.B) / n_el : 1.0f / n_el;
      const float* tg = p.target + (size_t)b * T * B2H_COUT;
      const float* cf = p.conf ? p.conf + (size_t)b * T * (B2H_COUT / 2) : nullptr;
      float* po = p.y ? p.y + (size_t)b * T * B2H_COUT : nullptr;
      float sum = 0.f;
      for (int i = threadIdx.x; i < T * B2H_COUT; i += kThreads) {
        const int t = i / B2H_COUT, co = i - t * B2H_COUT;
        float pr = G0[(t + 2) * ldg + co];
        float gr = 0.f;
        if (t >= len) {
          pr = 0.f;                                              // utils.py:311
        } else {
          const float tv = __ldg(tg + i);
          float d, s = 1.0f;
          if (p.loss_kind == B2H_LOSS_L1) {
            d = pr - tv;                                         // utils.py:422-426
          } else {
            s = __ldg(cf + t * (B2H_COUT / 2) + (co >> 1));
            d = __fsub_rn(__fmul_rn(pr, s), __fmul_rn(tv, s));   // utils.py:447-450
          }
          sum += fabsf(d);
          const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
          gr = sg * s * scale;
        }
        if (po) po[i] = pr;
        G0[(t + 2) * ldg + co] = gr;
      }
      const float tot = block_sum(sum, red);
      if (threadIdx.x == 0) loss_acc += tot / n_el;              // per-sample mean  utils.py:426 / :450
    } else {
      const float* dy = p.d_y + (size_t)b * T * B2H_COUT;
      for (int i = threadIdx.x; i < T * B2H_COUT; i += kThreads) {
        const int t = i / B2H_COUT, co = i - t * B2H_COUT;
        G0[(t + 2) * ldg + co] = __ldg(dy + i);
      }
    }
    __syncthreads();
    // layer 4: wgrad(dY, a3), dgrad -> dZ3 = (W4^T * dY) . (a3 > 0)
    wgrad_rows(G0, ldg, g.cout[3], A3, ldc, g.cin[3], part + g.w_off[3], part + g.b_off[3], T, first);
    conv_rows<2>(G0, ldg, g.cout[3], Wd[3], g.cin[3], nullptr, G1, ldg, A3, ldc, T);
    __syncthreads();
    wgrad_rows(G1, ldg, g.cout[2], A2, ldc, g.cin[2], part + g.w_off[2], part + g.b_off[2], T, first);
    conv_rows<2>(G1, ldg, g.cout[2], Wd[2], g.cin[2], nullptr, G0, ldg, A2, ldc, T);
    __syncthreads();
    wgrad_rows(G0, ldg, g.cout[1], A1, ldc, g.cin[1], part + g.w_off[1], part + g.b_off[1], T, first);
    conv_rows<2>(G0, ldg, g.cout[1], Wd[1], g.cin[1], nullptr, G1, ldg, A1, ldc, T);
    __syncthreads();
    wgrad_rows(G1, ldg, g.cout[0], X, ld0, g.cin[0], part + g.w_off[0], part + g.b_off[0], T, first);
    __syncthreads();
    first = false;
  }
  if (TRAIN && threadIdx.x == 0 && p.loss_partials) {
    // maskedPoseL1 divides by the batch size (utils.py:428); poderatedPoseL1 sums (utils.py:452)
    p.loss_partials[blockIdx.x] = (p.loss_kind == B2H_LOSS_L1) ? loss_acc / (float)p.B : loss_acc;
  }
}


FfmaPlan plan_ffma(const Geo& g, int B, int T, bool train) {
  FfmaPlan p{};
  p.train = train;
  const int TR = round_up(T, 8) + 4;
  const int ld0 = round_up(g.cin[0], 4), ldc = round_up(g.C, 4), ldg = round_up(g.C > B2H_COUT ? g.C : B2H_COUT, 4);
  size_t fl = train ? (size_t)TR * (ld0 + 3 * ldc + 2 * ldg) : (size_t)TR * (ld0 + 2 * ldc);
  p.smem = fl * 4;
  p.ok = p.smem <= (size_t)226 * 1024;   // dynamic + static shared memory must stay <= 227 KB
  int per_sm = 8;
  if (train) {
    per_sm = (int)((size_t)220 * 1024 / (p.smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 2) per_sm = 2;
  }
  const int cap = num_sms() * per_sm;
  p.grid = B < cap ? B : cap;
  return p;
}

int launch_fp32(const ConvArgs& a, const FfmaPlan& plan, cudaStream_t stream) {
  const void* fn = plan.train ? reinterpret_cast<const void*>(conv_fp32_kernel<true>) : reinterpret_cast<const void*>(conv_fp32_kernel<false>);
  // opt in to > 48 KB of dynamic shared memory
  if (int rc = ensure_dyn_smem(fn, plan.smem)) return rc;
  if (plan.train) conv_fp32_kernel<true><<<plan.grid, kThreads, plan.smem, stream>>>(a);
  else conv_fp32_kernel<false><<<plan.grid, kThreads, plan.smem, stream>>>(a);
  count_launch();
  return check_launch(plan.train ? "conv_fp32_kernel<train>" : "conv_fp32_kernel<fwd>");
}

}  // namespace b2h
