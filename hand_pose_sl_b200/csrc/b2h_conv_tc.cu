// bf16 mode (B2H_BF16): ConvModel forward as four fused implicit-GEMM layers on tcgen05 / TMEM.
//
// Reference semantics: ConvModel.forward  body2hand/src/models/HandPoseModels.py:40-64
//                      mask_output        body2hand/src/steps/utils.py:309-312
//
// Implicit GEMM without im2col.  A CTA owns G windows.  Their activations live in shared memory in
// "row space": [2 zero rows][window 0: T frames][2 zero rows][window 1]...[2 zero rows]; neighbouring
// windows share their zero padding, so the k=5 / pad=2 conv never sees another window's frames.
// A buffer is stored as [channel/8][row][8 channels] bf16 = the no-swizzle K-major UMMA canonical
// layout with 16-B rows: core matrix (8 rows x 16 B) contiguous, SBO = 128 B, LBO = rows*16 B.
// In that layout "tap k of output row r reads input row r+k-2" is just a +16*(k-2) byte change of the
// descriptor start address, so one layer for 128 output rows is 5 taps x (Cin/16) tcgen05.mma
// (M=128, N=Cout padded to 16, K=16) accumulating into one TMEM tile.  The epilogue
// (tcgen05.ld -> +bias -> ReLU -> bf16 -> st.shared) writes the next layer's A operand in place,
// forcing the shared zero rows back to 0; the last layer writes fp32 (B,T,42) to global.
#include "b2h_common.cuh"
#include "b2h_tc.cuh"

namespace b2h {
using namespace tc;

// ------------------------------------------------------------------------------------------------
// Probe: validates descriptor encodings, the row-shift trick, MN-major operands and the M=64 TMEM
// layout against a CPU matmul (tests/test_tc_probe.py).
//   mode 0: K-major.  D[m][n] = sum_k A[m+shift][k] * B[n][k]          A (136,K) B (N,K), M=128
//   mode 1: MN-major. D[m][n] = sum_t A[t][m] * B[t+shift][n]          A (K,128) B (K+8,N), M=128
//   mode 2: K-major, two M=64 MMAs: rows 0..63 -> TMEM lane 0, rows 64..127 -> TMEM lane 16;
//           out holds the raw 128 lanes x N columns.
// variant bit0: swap LBO/SBO, bit1: descriptor version field = 0.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) tc_probe_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ Bm,
                                                       float* __restrict__ out, int N, int ksteps, int shift, int variant,
                                                       int mode) {
  extern __shared__ __align__(128) unsigned char psm[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int K = 16 * ksteps;
  const int RA = (mode == 1) ? K : 136, CA = (mode == 1) ? 128 : K;
  const int RBm = (mode == 1) ? K + 8 : N, CB = (mode == 1) ? N : K;
  unsigned char* sa = psm;
  unsigned char* sb = psm + (size_t)(CA / 8) * RA * 16;
  // stage [c/8][r][8]
  for (int i = threadIdx.x; i < RA * CA; i += 128) {
    int r = i / CA, c = i - r * CA;
    *reinterpret_cast<__nv_bfloat16*>(sa + ((size_t)(c >> 3) * RA + r) * 16 + (c & 7) * 2) = A[i];
  }
  for (int i = threadIdx.x; i < RBm * CB; i += 128) {
    int r = i / CB, c = i - r * CB;
    *reinterpret_cast<__nv_bfloat16*>(sb + ((size_t)(c >> 3) * RBm + r) * 16 + (c & 7) * 2) = Bm[i];
  }
  if (threadIdx.x < 32) tmem_alloc(&tmem_slot, 256);
  if (threadIdx.x == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;
  const uint32_t ver = (variant & 2) ? 0u : 1u;
  if (threadIdx.x == 0) {
    const uint32_t a0 = smem_u32(sa), b0 = smem_u32(sb);
    for (int s = 0; s < ksteps; ++s) {
      if (mode == 0 || mode == 2) {
        uint32_t lboA = RA * 16, sboA = 128, lboB = RBm * 16, sboB = 128;
        if (variant & 1) { uint32_t t = lboA; lboA = sboA; sboA = t; t = lboB; lboB = sboB; sboB = t; }
        const uint64_t bd = make_smem_desc(b0 + (2 * s) * RBm * 16, lboB, sboB, ver);
        if (mode == 0) {
          const uint64_t ad = make_smem_desc(a0 + (2 * s) * RA * 16 + shift * 16, lboA, sboA, ver);
          umma_bf16(tbase, ad, bd, make_idesc_bf16(128, N, 0, 0), s > 0);
        } else {
          const uint64_t ad0 = make_smem_desc(a0 + (2 * s) * RA * 16 + shift * 16, lboA, sboA, ver);
          const uint64_t ad1 = make_smem_desc(a0 + (2 * s) * RA * 16 + (shift + 64) * 16, lboA, sboA, ver);
          umma_bf16(tbase, ad0, bd, make_idesc_bf16(64, N, 0, 0), s > 0);
          umma_bf16(tbase + (16u << 16), ad1, bd, make_idesc_bf16(64, N, 0, 0), s > 0);
        }
      } else {
        uint32_t lboA = 128, sboA = RA * 16, lboB = 128, sboB = RBm * 16;
        if (variant & 1) { uint32_t t = lboA; lboA = sboA; sboA = t; t = lboB; lboB = sboB; sboB = t; }
        const uint64_t ad = make_smem_desc(a0 + (16 * s) * 16, lboA, sboA, ver);
        const uint64_t bd = make_smem_desc(b0 + (16 * s + shift) * 16, lboB, sboB, ver);
        umma_bf16(tbase, ad, bd, make_idesc_bf16(128, N, 1, 1), s > 0);
      }
    }
    umma_commit(&bar);
  }
  __syncwarp();
  mbar_wait(&bar, 0, 1);
  tc_fence_after();
  const int warp = threadIdx.x >> 5;
  for (int c0 = 0; c0 < N; c0 += 16) {
    uint32_t v[16];
    tmem_ld16(tbase + ((uint32_t)(warp * 32) << 16) + c0, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 16; ++j) out[(size_t)threadIdx.x * N + c0 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tbase, 256);
}

// ------------------------------------------------------------------------------------------------
// Fused forward, v1: 128 threads (4 warps = the 4 TMEM lane quadrants); thread i owns output row i
// of every 128-row tile.  Layers run back to back out of shared memory.
// ------------------------------------------------------------------------------------------------


constexpr int kTcThreads = 128;
constexpr int kTileCols = 64;   // TMEM column stride between the accumulators of consecutive tiles

struct TcFwdArgs {
  const void* x; int x_dtype;
  const float* params; const char* packed; const int32_t* lengths;
  float* y;
  int B, T, G, NT, RBUF, apply_mask;
  float out_scale;
  Geo geo;
  WindowView wv;            // win_start set: x is a frame stream and B = the number of windows
};

__device__ __forceinline__ void store_row_bf16(unsigned char* buf, int chunk_stride, int row, int c0, const float* v8) {
  uint4 q;
  q.x = pack_bf16x2(v8[0], v8[1]); q.y = pack_bf16x2(v8[2], v8[3]);
  q.z = pack_bf16x2(v8[4], v8[5]); q.w = pack_bf16x2(v8[6], v8[7]);
  *reinterpret_cast<uint4*>(buf + (size_t)(c0 >> 3) * chunk_stride + (size_t)row * 16) = q;
}

__global__ void __launch_bounds__(kTcThreads, 1) conv_tc_fwd_kernel(TcFwdArgs p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  __shared__ float bias_s[4][64];
  const Geo& g = p.geo;
  const int T = p.T, G = p.G, NT = p.NT, RBUF = p.RBUF;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int b0 = blockIdx.x * G;
  const int CH = RBUF * 16;                       // byte stride between 8-channel chunks
  const int KPmax = g.kp[0] > g.kp[1] ? g.kp[0] : g.kp[1];
  const int buf_bytes = (KPmax / 8) * CH;
  // smem carve: [weights l0..l3][buf0][buf1]
  int w_bytes[4], w_off[4], wtot = 0;
#pragma unroll
  for (int l = 0; l < 4; ++l) { w_off[l] = wtot; w_bytes[l] = B2H_KW * g.kp[l] * g.np_[l] * 2; wtot += w_bytes[l]; }
  unsigned char* wsm = smem;
  unsigned char* buf0 = smem + ((wtot + 127) / 128) * 128;
  unsigned char* buf1 = buf0 + buf_bytes;

  uint32_t ncols = 32;
  while ((int)ncols < NT * kTileCols) ncols <<= 1;
  if (warp == 0) tmem_alloc(&tmem_slot, ncols);
  if (tid == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  // weights: packed bf16 UMMA blocks, contiguous per layer
  for (int l = 0; l < 4; ++l) {
    const uint4* src = reinterpret_cast<const uint4*>(p.packed + g.tf_off[l]);
    uint4* dst = reinterpret_cast<uint4*>(wsm + w_off[l]);
    for (int i = tid; i < w_bytes[l] / 16; i += kTcThreads) dst[i] = __ldg(src + i);
  }
  for (int i = tid; i < 4 * 64; i += kTcThreads) {
    const int l = i >> 6, c = i & 63;
    bias_s[l][c] = (c < g.cout[l]) ? __ldg(p.params + g.b_off[l] + c) : 0.0f;
  }
  {  // zero both activation buffers (padding rows / channels stay zero for the whole kernel)
    uint4* z = reinterpret_cast<uint4*>(buf0);
    const uint4 zero = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < 2 * buf_bytes / 16; i += kTcThreads) z[i] = zero;
  }
  __syncthreads();
  // stage the input windows: (T, n_in) NWC -> buf0 rows, bf16.  Source row of (window b, frame t): b*T + t, or the window
  // view's decode (-1: a zero row, left as zeroed above; the pos-emb channel is written for it all the same)
  {
    const int n_in = g.n_in, pe = g.pos_emb;
    const int nwin = (p.B - b0) < G ? (p.B - b0) : G;
    auto src_row = [&](int b, int t) -> long long { return p.wv.win_start ? window_src_row(p.wv, b, t) : (long long)b * T + t; };
    if (pe == 0 && (n_in & 7) == 0) {
      const int cpr = n_in >> 3;                 // 16-B chunks per row
      for (int i = tid; i < nwin * T * cpr; i += kTcThreads) {
        const int c8 = i % cpr, ft = i / cpr;
        const int gi = ft / T, t = ft - gi * T;
        const int row = 2 + gi * (T + 2) + t;
        const long long sr = src_row(b0 + gi, t);
        if (sr < 0) continue;
        float v[8];
        if (p.x_dtype == B2H_DT_F32) {
          const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.x) + (size_t)sr * n_in + c8 * 8);
          const float4 lo = __ldg(src), hi = __ldg(src + 1);
          v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
          store_row_bf16(buf0, CH, row, c8 * 8, v);
        } else {
          const uint4 q = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.x) + (size_t)sr * n_in + c8 * 8));
          *reinterpret_cast<uint4*>(buf0 + (size_t)c8 * CH + (size_t)row * 16) = q;
        }
      }
    } else {
      for (int i = tid; i < nwin * T * n_in; i += kTcThreads) {
        const int c = i % n_in, ft = i / n_in;
        const int gi = ft / T, t = ft - gi * T;
        const int row = 2 + gi * (T + 2) + t;
        const long long sr = src_row(b0 + gi, t);
        if (sr < 0) continue;
        const size_t gidx = (size_t)sr * n_in + c;
        const float v = (p.x_dtype == B2H_DT_F32) ? __ldg(reinterpret_cast<const float*>(p.x) + gidx)
                                                  : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.x)[gidx]);
        const int cc = c + pe;
        *reinterpret_cast<__nv_bfloat16*>(buf0 + (size_t)(cc >> 3) * CH + (size_t)row * 16 + (cc & 7) * 2) = __float2bfloat16_rn(v);
      }
      if (pe) {  // LinearPositionalEmbedding channel 0 = t/100   HandPoseModels.py:70-82
        for (int i = tid; i < nwin * T; i += kTcThreads) {
          const int gi = i / T, t = i - gi * T;
          const int row = 2 + gi * (T + 2) + t;
          *reinterpret_cast<__nv_bfloat16*>(buf0 + (size_t)row * 16) = __float2bfloat16_rn(__fdiv_rn((float)t, (float)g.pe_len));
        }
      }
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;
  uint32_t phase = 0;

  for (int l = 0; l < 4; ++l) {
    unsigned char* bin = (l & 1) ? buf1 : buf0;
    unsigned char* bout = (l & 1) ? buf0 : buf1;
    const int KS = g.kp[l] >> 4, N = g.np_[l];
    if (tid == 0) {
      const uint32_t idesc = make_idesc_bf16(128, N, 0, 0);
      const uint32_t a_base = smem_u32(bin), w_base = smem_u32(wsm + w_off[l]);
      for (int j = 0; j < NT; ++j) {
        uint32_t acc = 0;
        for (int k = 0; k < B2H_KW; ++k) {
          for (int s = 0; s < KS; ++s) {
            // output row r = 2+128j+i reads input row r+k-2 = 128j+k+i
            const uint64_t ad = make_smem_desc(a_base + (2 * s) * CH + (128 * j + k) * 16, CH, 128);
            const uint64_t bd = make_smem_desc(w_base + (k * KS + s) * (N * 32), N * 16, 128);
            umma_bf16(tbase + j * kTileCols, ad, bd, idesc, acc);
            acc = 1;
          }
        }
      }
      umma_commit(&bar);
    }
    __syncwarp();
    mbar_wait(&bar, phase, 10 + l);
    phase ^= 1;
    tc_fence_after();
    for (int j = 0; j < NT; ++j) {
      const int row = 2 + 128 * j + tid;
      const int rel = row - 2;
      const int gi = rel / (T + 2), t = rel - gi * (T + 2);
      const bool valid = (t < T) && (gi < G) && (b0 + gi < p.B);
      const uint32_t taddr = tbase + ((uint32_t)(warp * 32) << 16) + j * kTileCols;
      if (l < 3) {
        for (int c0 = 0; c0 < N; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
          float f[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) f[q] = valid ? fmaxf(__uint_as_float(v[q]) + bias_s[l][c0 + q], 0.0f) : 0.0f;
          store_row_bf16(bout, CH, row, c0, f);
          store_row_bf16(bout, CH, row, c0 + 8, f + 8);
        }
      } else {
        int len = T;
        if (valid && p.lengths) { len = p.lengths[b0 + gi]; }
        float* yrow = valid ? p.y + ((size_t)(b0 + gi) * T + t) * B2H_COUT : nullptr;
        for (int c0 = 0; c0 < N; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);      // warp-collective: every lane must execute it
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int q = 0; q < 16; q += 2) {
              const int c = c0 + q;
              if (c < B2H_COUT) {
                float a = __uint_as_float(v[q]) + bias_s[3][c];
                float b = __uint_as_float(v[q + 1]) + bias_s[3][c + 1];
                if (p.apply_mask && t >= len) { a = 0.0f; b = 0.0f; }        // mask_output utils.py:309-312
                else if (p.out_scale != 1.0f) { a *= p.out_scale; b *= p.out_scale; }
                *reinterpret_cast<float2*>(yrow + c) = make_float2(a, b);
              }
            }
          }
        }
      }
    }
    fence_proxy_async_smem();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (warp == 0) tmem_dealloc(tbase, ncols);
}


// G = enough windows per CTA to cover B with one CTA per SM, capped by the row space (<= 8 tiles of 128 rows) and by the
// 225 KB of shared memory that hold all four layers' weights and two activation buffers of RBUF rows.
RowspacePlan plan_rowspace(const Geo& g, int B, int T) {
  RowspacePlan p{};
  int wtot = 0;
  for (int l = 0; l < 4; ++l) wtot += B2H_KW * g.kp[l] * g.np_[l] * 2;
  const int KPmax = g.kp[0] > g.kp[1] ? g.kp[0] : g.kp[1];
  auto geometry = [&](int G) {
    p.G = G;
    p.NT = (G * (T + 2) - 2 + 127) / 128;
    p.RBUF = 128 * p.NT + 8;
    p.smem = (size_t)((wtot + 127) / 128) * 128 + (size_t)2 * (KPmax / 8) * p.RBUF * 16;
  };
  if (g.C > 64 || g.cin[0] > 64 || T < 1 || T > 8 * 128) return p;
  const int sms = num_sms();
  int G = (B + sms - 1) / sms;
  const int gmax = (8 * 128 + 2) / (T + 2);
  if (G > gmax) G = gmax;
  if (G < 1) G = 1;
  geometry(G);
  while (p.G > 1 && p.smem > (size_t)225 * 1024) geometry(p.G - 1);
  p.ok = p.smem <= (size_t)225 * 1024;
  p.grid = (B + p.G - 1) / p.G;
  return p;
}

int launch_tc_fwd(const ConvArgs& a, const RowspacePlan& plan, cudaStream_t stream) {
  TcFwdArgs p{};
  p.x = a.x; p.x_dtype = a.x_dtype; p.params = a.params; p.packed = a.packed; p.lengths = a.lengths;
  p.y = a.y; p.B = a.B; p.T = a.T; p.apply_mask = a.apply_mask; p.out_scale = a.out_scale; p.geo = a.geo; p.wv = a.wv;
  p.G = plan.G; p.NT = plan.NT; p.RBUF = plan.RBUF;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_tc_fwd_kernel), plan.smem)) return rc;
  conv_tc_fwd_kernel<<<plan.grid, kTcThreads, plan.smem, stream>>>(p);
  count_launch();
  return check_launch("conv_tc_fwd_kernel");
}

int launch_tc_probe(const void* a, const void* b, float* out, int n, int ksteps, int shift, int variant, cudaStream_t stream) {
  const int mode = variant >> 4;
  variant &= 15;
  if (n % 16 || n < 16 || n > 256 || ksteps < 1 || ksteps > 8 || shift < 0 || shift > 8 || mode < 0 || mode > 2) {
    set_error("b2h_tc_probe: bad arguments");
    return B2H_EINVAL;
  }
  const int K = 16 * ksteps;
  const size_t bytes = (mode == 1) ? (size_t)16 * K * 16 + (size_t)(n / 8) * (K + 8) * 16 : (size_t)(K / 8) * 136 * 16 + (size_t)(K / 8) * n * 16;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(tc_probe_kernel), 200 * 1024)) return rc;
  tc_probe_kernel<<<1, 128, bytes + 128, stream>>>(reinterpret_cast<const __nv_bfloat16*>(a), reinterpret_cast<const __nv_bfloat16*>(b), out, n,
                                                   ksteps, shift, variant, mode);
  count_launch();
  return check_launch("tc_probe_kernel");
}

int tc_status_and_clear() {
  int v = 0, z = 0;
  cudaMemcpyFromSymbol(&v, g_tc_status, sizeof(int));
  if (v) {
    cudaMemcpyToSymbol(g_tc_status, &z, sizeof(int));
    cudaMemcpyToSymbol(g_dp_abort, &z, sizeof(int));
  }
  return v;
}

}  // namespace b2h

namespace b2h {
using namespace tc;
// ------------------------------------------------------------------------------------------------
// Microbenchmark (bring-up aid): cycles per tcgen05.mma for a given shape, issued back to back by one
// thread, rotating over `nacc` accumulators.  out[0] = cycles from first issue to completion,
// out[1] = cycles spent in the issue loop alone.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) tc_bench_kernel(long long* out, int M, int N, int reps, int nacc, int mn_major, int rows) {
  extern __shared__ __align__(128) unsigned char bsm[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  __shared__ __align__(8) uint64_t bar2;
  const bool rnd = (mn_major >> 4) & 1;          // non-zero operand bits (values in [1, 2)): data-dependent pacing / power
  for (int i = tid; i < 64 * 1024 / 16; i += 128) {
    uint32_t h = (uint32_t)i * 2654435761u + blockIdx.x * 40503u;
    const uint32_t w0 = rnd ? (0x3F803F80u | (h & 0x007F007Fu)) : 0u, w1 = rnd ? (0x3F803F80u | ((h >> 7) & 0x007F007Fu)) : 0u;
    reinterpret_cast<uint4*>(bsm)[i] = make_uint4(w0, w1, w0 ^ (rnd ? 0x00150015u : 0u), w1 ^ (rnd ? 0x002A002Au : 0u));
  }
  if (warp == 0) tmem_alloc(&tmem_slot, 512);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;
  long long t0 = 0, t1 = 0;
  const int nissue = nacc >> 8;          // upper bits: number of issuing warps (each with its own accumulators)
  nacc &= 255;
  if (tid == 0) { mbar_init(&bar, nissue > 0 ? nissue : 1); mbar_init(&bar2, 1u << 20); fence_barrier_init(); }
  __syncthreads();
  if (warp < (nissue > 0 ? nissue : 1)) {
    if (elect_one()) {
      const uint32_t a0 = smem_u32(bsm), b0 = smem_u32(bsm + 32 * 1024);
      const uint32_t CH = rows * 16;
      const int vary = (mn_major >> 2) & 1;    // walk A rows and B blocks like a streamed-weight main loop
      const int commit2 = (mn_major >> 3) & 1; // tcgen05.commit after every second MMA (ring-stage release)
      const int sw128 = (mn_major >> 1) & 1;   // timing-only variant: 128-byte-swizzle K-major descriptors (SBO = 1024 B)
      mn_major &= 1;
      uint64_t ad = mn_major ? make_smem_desc(a0, 128, CH) : make_smem_desc(a0, CH, 128);
      uint64_t bd = mn_major ? make_smem_desc(b0, 128, CH) : make_smem_desc(b0, CH, 128);
      if ((mn_major >> 5) & 1) bd = make_smem_desc(b0, 4096, 128);   // B chunk stride = even multiple of 128 B
      if ((mn_major >> 6) & 1) ad = make_smem_desc(a0, 4096, 128);   // A chunk stride likewise
      if ((mn_major >> 7) & 1) bd = make_smem_desc(b0, 4096 + 128, 128);
      if (sw128) {
        ad = make_smem_desc(a0, 16, 1024) | (2ull << 61);
        bd = make_smem_desc(b0, 16, 1024) | (2ull << 61);
      }
      const uint32_t idesc = make_idesc_bf16(M, N, mn_major, mn_major);
      const uint32_t dbase = tbase + warp * nacc * N;
      t0 = clock64();
      if (!vary && !commit2) {
        for (int r = 0; r < reps; ++r) umma_bf16(dbase + (r % nacc) * N, ad + (uint64_t)(sw128 ? 2 * (r & 3) : (r & 3)), bd, idesc, 1);
      } else {
        for (int r = 0; r < reps; ++r) {
          const uint64_t aoff = vary ? (uint64_t)(((r >> 1) * 7) & 63) + (uint64_t)((r & 1) * 128) : (uint64_t)(r & 3);
          const uint64_t boff = vary ? (uint64_t)(((r >> 1) & 3) * 256) : 0ull;      // 4-KB steps
          umma_bf16(dbase + (r % nacc) * N, ad + aoff, bd + boff, idesc, 1);
          if (commit2 && (r & 1)) umma_commit(&bar2);
        }
      }
      t1 = clock64();
      umma_commit(&bar);
    }
    __syncwarp();
  }
  mbar_wait(&bar, 0, 40);
  const long long t2 = clock64();
  if (warp == 0 && t0 != 0 && blockIdx.x == 0) { out[0] = t2 - t0; out[1] = t1 - t0; }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, 512);
}

// Bring-up microbenchmark (M == 1 in b2h_tc_bench): steady-state global(L2) -> shared throughput of 1-D bulk copies.
// A ring of `depth` 8-KB stages is kept full by one warp; every stage is fetched as 8192/copy_bytes copies issued by
// consecutive lanes.  out[0] = cycles, out[1] = bytes moved (CTA 0).
__device__ unsigned char g_tma_src[1 << 20];
__global__ void __launch_bounds__(32) tma_bench_kernel(long long* out, int copy_bytes, int rounds, int depth) {
  extern __shared__ __align__(128) unsigned char bsm[];
  __shared__ __align__(8) uint64_t full[16];
  const int lane = threadIdx.x;
  if (lane == 0) { for (int s = 0; s < depth; ++s) mbar_init(&full[s], 1); fence_barrier_init(); }
  __syncwarp();
  const int ncopy = 8192 / copy_bytes;
  auto issue = [&](int s, int blk) {
    if (lane == 0) mbar_arrive_expect_tx(&full[s], 8192);
    __syncwarp();
    for (int c = lane; c < ncopy; c += 32)
      bulk_g2s(bsm + s * 8192 + c * copy_bytes, g_tma_src + (size_t)(blk & 127) * 8192 + c * copy_bytes, copy_bytes, &full[s]);
  };
  int blk = 0;
  for (int s = 0; s < depth; ++s) issue(s, blk++);
  const long long t0 = clock64();
  for (int r = 0; r < rounds; ++r)
    for (int s = 0; s < depth; ++s) {
      mbar_wait(&full[s], r & 1, 41);
      __syncwarp();
      issue(s, blk++);
    }
  const long long t1 = clock64();
  for (int s = 0; s < depth; ++s) mbar_wait(&full[s], rounds & 1, 42);
  if (lane == 0 && blockIdx.x == 0) { out[0] = t1 - t0; out[1] = (long long)rounds * depth * 8192; }
}

int launch_tc_bench(long long* out, int M, int N, int reps, int nacc, int mn_major, cudaStream_t stream) {
  if (M == 1) {   // TMA bulk-copy throughput: N = bytes per copy, reps = rounds, nacc = ring depth, mn_major = CTAs
    if (N < 16 || N > 8192 || (8192 % N) || nacc < 1 || nacc > 16 || reps < 1 || mn_major < 1) { set_error("b2h_tc_bench(tma): bad arguments"); return B2H_EINVAL; }
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(tma_bench_kernel), 128 * 1024)) return rc;
    tma_bench_kernel<<<mn_major, 32, 128 * 1024, stream>>>(out, N, reps, nacc);
    count_launch();
    return check_launch("tma_bench_kernel");
  }
  if ((M != 64 && M != 128) || N < 8 || N > 256 || (N % (M == 64 ? 8 : 16)) || reps < 1 || (nacc & 255) < 1 || (nacc & 255) * N * ((nacc >> 8) > 0 ? (nacc >> 8) : 1) > 512 || (nacc >> 8) > 4) {
    set_error("b2h_tc_bench: bad arguments");
    return B2H_EINVAL;
  }
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(tc_bench_kernel), 64 * 1024)) return rc;
  const int grid = (mn_major >> 8) > 0 ? (mn_major >> 8) : 1;     // bits 8..: CTAs (all SMs busy -> chip-level pacing)
  tc_bench_kernel<<<grid, 128, 64 * 1024, stream>>>(out, M, N, reps, nacc, mn_major & 255, 136);
  count_launch();
  return check_launch("tc_bench_kernel");
}
}  // namespace b2h

#include "b2h_train_tc.cuh"
#include "b2h_wide_tc.cuh"
