// bf16 mode, wide forward kernel (64 < conv_channels <= 256): ConvModel.forward on tcgen05 / TMEM with the weights
// STREAMED through shared memory.  Included by b2h_conv_tc.cu (same translation unit as the PTX layer).
//
// Reference semantics: ConvModel.forward  body2hand/src/models/HandPoseModels.py:40-64 (`--conv-channels`, run.py),
//                      mask_output        body2hand/src/steps/utils.py:309-312 (optional epilogue).
//
// At C = 256 one layer's weights are 5 x 256 x 256 bf16 = 640 KB: they cannot live in shared memory like the C <= 64
// tile kernel's (b2h_train_tc.cuh), and an N = 256 MMA is datapath-bound (128 x 256 x 16 MACs = 128 tensor cycles)
// instead of instruction-bound.  So the kernel is organised like a GEMM main loop:
//   * tile = 256 output rows = two M=128 accumulators of N <= 256 fp32 columns = all 512 TMEM columns; the rows hold
//     floor(258 / (T+2)) whole windows separated by 2 shared zero rows (T=64: 3 windows, T=126: 2, T<=256: 1);
//   * ONE activation buffer [channel/8][264 rows][8 ch] bf16 (no-swizzle K-major UMMA layout, conv tap k = +k rows in
//     the descriptor start address) that every layer reads and then overwrites IN PLACE: all MMAs of a layer have
//     completed (commit -> acc_full) before its epilogue writes, and inference keeps no activations;
//   * the packed UMMA B blocks (b2h_common.cuh umma_b_offset: one [2][N][8] block per (tap, 16-channel k-step),
//     contiguous in global memory) stream through a ring of 16-KB stages by TMA tensor-map loads (the packed sections
//     viewed as a 2-D tensor of 128-byte rows, box = 128 rows; measured here: 1-D cp.async.bulk copies top out at
//     ~23 B/cycle/SM, a third of what two N=256 MMAs per stage consume) issued by a dedicated producer warp that
//     runs ahead across layers and tiles; full[]/empty[] mbarriers, the empty side armed by tcgen05.commit of the
//     MMAs that read the stage;
//   * warp roles: 8 epilogue warps (two per TMEM lane quadrant, alternating 32-column chunks: tcgen05.ld -> bias/ReLU
//     -> bf16 -> st.shared, or the fp32 prediction rows of layer 4), 1 MMA-issuing warp, 1 weight-producer warp.
#pragma once
#include <cuda.h>   // CUtensorMap + enums only; the encoder is fetched with cudaGetDriverEntryPoint (no libcuda link)

namespace b2h {
using namespace tc;

// One GEMM stage of the wide kernels: a conv layer (forward) or a dgrad layer (backward): K = 16*KS reduction channels,
// N output channels, blocks streamed from 128-byte row `row0` of the weight tensor map.
struct WideStageDesc { int KS, N, row0, layer; };

struct WideArgs {
  const void* x; int x_dtype;
  const float* params; const char* packed; const int32_t* lengths;
  float* y;
  long long* dbg;
  int B, T, apply_mask;
  float out_scale;
  int n_tiles, gh, nstage, a_bytes;
  Geo geo;
  int n_stages;                 // 4 conv layers (forward) / 3 dgrad layers (backward chain)
  WideStageDesc st[4];
  // training (MODE 1: forward that saves every layer input + criterion; MODE 2: dgrad chain)
  const float* target; const float* conf; const float* d_y;
  int loss_kind, train_mode;    // train_mode 1 = criterion inside, 2 = backward of a given d_y
  unsigned char* scratch;       // per tile: the layer inputs ACT[0..3] and the pre-activation gradients DZ[0..3], each a
  long long tile_bytes;         // dump of the shared-memory operand layout [channel/8][264 rows][8 ch] bf16
  long long act_off[4], dz_off[4];
  float* loss_partials;         // [grid]
  long long* step_dev; long long* epoch_dev;   // MODE 1: device-side step / exchange-epoch counters, bumped by CTA 0 (read by the Adam kernel)
  WindowView wv;                // MODE 0 / 1: win_start set = x (and target / conf) are frame streams, B = windows viewed in them
};

constexpr int kWideThreads = 320;
constexpr int kWideEpiThreads = 256;
constexpr int kWideRows = 264;            // 2 zero rows + 256 output rows + 6 zero rows
constexpr int kWideStage = 16384;         // bytes per ring stage (two N=256 blocks, or several narrower ones)
constexpr int kWideBoxRows = kWideStage / 128;
constexpr int kWideMaxStages = 16;

struct WideSched { int KS, N, blk_bytes, nblk, bps, nst; };
__host__ __device__ inline WideSched wide_sched(int KS, int N) {
  WideSched s;
  s.KS = KS; s.N = N;
  s.blk_bytes = s.N * 32;
  s.nblk = B2H_KW * s.KS;
  s.bps = kWideStage / s.blk_bytes; if (s.bps < 1) s.bps = 1;
  s.nst = (s.nblk + s.bps - 1) / s.bps;
  return s;
}

// scratch layout of one tile for wide training (byte offsets; every dump = chunks x kWideRows x 16 B)
struct WideScratch { long long act_off[4], dz_off[4], tile_bytes; };
__host__ __device__ inline WideScratch wide_scratch(const Geo& g) {
  WideScratch w;
  long long o = 0;
  const long long CHB = (long long)kWideRows * 16;
  for (int l = 0; l < 4; ++l) { w.act_off[l] = o; o += (g.kp[l] / 8) * CHB; }       // input of layer l
  for (int l = 0; l < 4; ++l) { w.dz_off[l] = o; o += (g.np_[l] / 8) * CHB; }       // dZ_l (padded output channels of layer l)
  w.tile_bytes = o;
  return w;
}

// raw shared-address variants of the barrier / TMA / commit helpers for the two single-thread loops
__device__ __forceinline__ void tma_load_2d_addr(uint32_t smem_dst, const CUtensorMap* tmap, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(smem_dst), "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void expect_tx_addr(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void commit_addr(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool wait_addr(uint32_t bar, uint32_t parity, int site) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  if (ok) return true;                               // fast path: no clock reads
  const long long t0 = clock64();
  for (;;) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return true;
    if (clock64() - t0 > 4000000000LL) { atomicExch(&g_tc_status, site); return false; }
  }
}

// MODE 0: inference forward (ConvModel.forward, optional mask_output / de-normalise epilogue).
// MODE 1: training forward: the same four layers, every layer INPUT (x, a1, a2, a3) is also written to the tile's scratch
//         dump in the shared-memory operand layout, and the layer-4 epilogue is the criterion: masked prediction,
//         maskedPoseL1 / poderatedPoseL1 term, d(loss)/d(pred) -> DZ[3] (steps/utils.py:309-312, 413-452).
// MODE 2: dgrad chain: DZ[3] -> DZ[2] -> DZ[1] -> DZ[0] with the transposed weight blocks; epilogue = ReLU mask on the
//         saved activation (loss.backward(), steps/traintest.py:120).  The weight gradients are a separate split-K GEMM
//         over the dumps (conv_tc_wide_wgrad_kernel).
// VIEW (MODE 1 only): training over window views, a separate instantiation so that the dense training forward keeps its
// code (the run-time test cost the C = 256 step ~0.6 %).  MODE 0 tests p.wv.win_start at run time.
template <int MODE, bool VIEW = false>
__global__ void __launch_bounds__(kWideThreads, 1) conv_tc_wide_kernel(WideArgs p, const __grid_constant__ CUtensorMap wmap) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full_bar[kWideMaxStages];    // stage landed (TMA complete_tx)
  __shared__ __align__(8) uint64_t empty_bar[kWideMaxStages];   // stage consumed (tcgen05.commit)
  __shared__ __align__(8) uint64_t acc_full;                    // a layer's accumulators are complete
  __shared__ __align__(8) uint64_t act_ready;                   // activation buffer written + accumulators drained
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float bias_s[4][256];
  __shared__ float loss_w[8];
  const Geo& g = p.geo;
  const int T = p.T, gh = p.gh;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  constexpr int rows = kWideRows;
  constexpr int CH = rows * 16;
  unsigned char* A = smem;
  unsigned char* RING = smem + p.a_bytes;
  const int S = p.nstage;
  const int NL = p.n_stages;

  // ---- setup: biases, zeroed activation buffer, barriers, TMEM ----
  for (int i = tid; i < 4 * 256; i += kWideThreads) {
    const int l = i >> 8, c = i & 255;
    bias_s[l][c] = c < g.cout[l] ? __ldg(p.params + g.b_off[l] + c) : 0.0f;
  }
  {
    uint4* z = reinterpret_cast<uint4*>(A);
    const uint4 zero = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < p.a_bytes / 16; i += kWideThreads) z[i] = zero;
  }
  if (warp == 0) tmem_alloc(&tmem_slot, 512);
  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&acc_full, 1);
    mbar_init(&act_ready, kWideEpiThreads);
    fence_barrier_init();
    if (MODE == 1 && blockIdx.x == 0) {
      if (p.step_dev) *p.step_dev += 1;
      if (p.epoch_dev) *p.epoch_dev += 1;
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;

  // Both single-thread loops below are latency-bound scalar code (every instruction waits for the previous one): a
  // first version that recomputed slot = stage % S, the barrier addresses and the descriptors per stage needed ~540
  // cycles per stage -- twice the 258 tensor cycles of the two N=256 MMAs it feeds.  So: raw shared-memory addresses
  // computed once, ring position and parity carried as counters, descriptors advanced by one add.
  const uint32_t full0 = smem_u32(&full_bar[0]), empty0 = smem_u32(&empty_bar[0]), ring0 = smem_u32(RING);
  if (warp == 9) {
    // ===================== weight producer: one thread, runs ahead by the ring depth =====================
    if (elect_one()) {
      uint32_t slot = 0, ph = 1;                     // parity 1 on a fresh barrier = "already free" (first lap)
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x)
        for (int l = 0; l < NL; ++l) {
          const WideSched sc = wide_sched(p.st[l].KS, p.st[l].N);
          int row = p.st[l].row0;                                        // 128-byte rows of the weight tensor map
          const int rows_per_stage = (sc.bps * sc.blk_bytes) >> 7;
          for (int st = 0; st < sc.nst; ++st) {
            if (!wait_addr(empty0 + slot * 8, ph, 60)) return;
            // one 128-row box = 16 KB whatever the stage's payload is (rows past it belong to the next stage / are
            // zero-filled past the tensor): the transaction count is always the full box
            expect_tx_addr(full0 + slot * 8, kWideStage);
            tma_load_2d_addr(ring0 + slot * kWideStage, &wmap, 0, row, full0 + slot * 8);
            row += rows_per_stage;
            if (++slot == (uint32_t)S) { slot = 0; ph ^= 1; }
          }
        }
    }
    __syncwarp();
  } else if (warp == 8) {
    // ===================== MMA issuer: one thread =====================
    if (elect_one()) {
      uint32_t slot = 0, ph = 0, act_phase = 0;
      int dn = 0;
      const uint32_t hi_k = desc_hi(128);
      const uint32_t a_lo0 = desc_lo(smem_u32(A), (uint32_t)CH);
      const uint32_t acc_addr = smem_u32(&acc_full);
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x)
        for (int l = 0; l < NL; ++l) {
          const WideSched sc = wide_sched(p.st[l].KS, p.st[l].N);
          const uint32_t idesc = make_idesc_bf16(128, sc.N, 0, 0);
          const uint32_t b_lo0 = desc_lo(ring0, (uint32_t)sc.N * 16);   // + slot * stage + block * blk, in 16-B units
          const uint32_t blk16 = (uint32_t)sc.blk_bytes >> 4;
          if (!mbar_wait(&act_ready, act_phase, 61)) return;
          act_phase ^= 1;
          tc_fence_after();
          if (p.dbg && blockIdx.x == 0 && dn < 8) p.dbg[dn++] = clock64();   // layer inputs ready
          if (MODE != 0) {
            // Training: the buffer now holds this stage's INPUT, which the weight-gradient GEMM needs later: dump it to the
            // tile's scratch with asynchronous bulk stores (TMA engine) that run under this stage's MMAs.  MODE 1: ACT[l]
            // (x, a1, a2, a3).  MODE 2: the input of stage j > 0 is the previous stage's output dZ -> DZ[layer] (DZ[3] was
            // written by the forward's criterion epilogue; the last stage's output DZ[0] is stored by its epilogue threads).
            // The epilogue threads ran fence.proxy.async before arriving on act_ready.
            const int nch = MODE == 1 ? g.kp[l] / 8 : g.np_[p.st[l].layer] / 8;
            if (MODE == 1 || l > 0) {
              unsigned char* dst = p.scratch + (size_t)tile * p.tile_bytes + (MODE == 1 ? p.act_off[l] : p.dz_off[p.st[l].layer]);
              for (int c = 0; c < nch; c += 4) {
                const int n = nch - c < 4 ? nch - c : 4;
                bulk_s2g(dst + (size_t)c * CH, A + (size_t)c * CH, (uint32_t)n * CH);
              }
              bulk_commit();
            }
          }
          int s = 0, left = sc.nblk;
          uint32_t a_tap = a_lo0, a_cur = a_lo0;       // output row 2+m reads input row m+k: tap k = +k rows
          uint32_t acc = 0;
          for (int st = 0; st < sc.nst; ++st) {
            // no tcgen05.fence after this wait: the mbarrier orders the TMA writes before the MMAs' reads
            if (!wait_addr(full0 + slot * 8, ph, 62)) return;
            uint32_t b_cur = b_lo0 + slot * (kWideStage >> 4);
            const int nb = left < sc.bps ? left : sc.bps;
            left -= nb;
            for (int b = 0; b < nb; ++b) {
              const uint64_t bd = desc64(b_cur, hi_k);
              umma_bf16(tbase, desc64(a_cur, hi_k), bd, idesc, acc);
              umma_bf16(tbase + 256, desc64(a_cur + 128, hi_k), bd, idesc, acc);
              acc = 1;
              b_cur += blk16;
              a_cur += 2 * rows;                       // next 16-channel k-step: two chunks further
              if (++s == sc.KS) { s = 0; a_tap += 1; a_cur = a_tap; }
            }
            commit_addr(empty0 + slot * 8);            // stage reusable once these MMAs have read it
            if (++slot == (uint32_t)S) { slot = 0; ph ^= 1; }
          }
          if (MODE != 0) bulk_wait_read0();            // the dump has read the buffer: the epilogue may overwrite it in place
          commit_addr(acc_addr);
          if (p.dbg && blockIdx.x == 0 && dn < 8) p.dbg[dn++] = clock64();   // layer MMAs issued
        }
      if (MODE != 0) bulk_wait0();                     // every dump has reached global memory before the CTA retires
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (256 threads): staging, bias/ReLU, prediction rows =====================
    const int r128 = tid & 127;
    const int ch = warp >> 2;                                  // column half (alternating 32-column chunks)
    const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
    const int n_in = g.n_in, pe = g.pos_emb;
    const int nch0 = g.kp[0] / 8;
    const bool vec_in = (pe == 0) && ((n_in & 7) == 0);
    float loss_run = 0.0f;                                     // MODE 1: this thread's share of the criterion
    struct RowCtx { int row, t, gw; bool valid; };
    auto rowctx = [&](int j, int tile) {
      const int mm = r128 + 128 * j;
      const int wjj = mm / (T + 2);
      RowCtx r;
      r.t = mm - wjj * (T + 2);
      r.row = 2 + mm;
      r.gw = tile * gh + wjj;
      r.valid = (r.t < T) && (wjj < gh) && (r.gw < p.B) && tile < p.n_tiles;
      return r;
    };
    // scratch dumps of tile `tile` (training): same [chunk][row][8 ch] layout as the shared-memory buffer
    auto dump = [&](int tile, long long off) { return p.scratch + (size_t)tile * p.tile_bytes + off; };
    auto zero_halo = [&](unsigned char* d, int nchunks) {      // rows 0,1 and 258..263 of every chunk are never written by rows
      const int et = tid;                                      // 0..255
      for (int i = et; i < nchunks * 8; i += kWideEpiThreads) {
        const int c = i >> 3, h = i & 7;
        const int row = h < 2 ? h : 256 + h;
        *reinterpret_cast<uint4*>(d + (size_t)c * CH + (size_t)row * 16) = make_uint4(0, 0, 0, 0);
      }
    };
    auto stage_inputs = [&](int tile) {      // (n_in) channels NWC -> chunks [0, kp0/8) of the activation buffer
      if (MODE == 2) {                       // backward chain: the tile's dZ_4 dump (criterion gradient) -> chunks [0, np4/8)
        if (tile >= p.n_tiles) return;
        const int nch = g.np_[3] / 8;
        const uint4* src = reinterpret_cast<const uint4*>(dump(tile, p.dz_off[3]));
        uint4* dst = reinterpret_cast<uint4*>(A);
        for (int i = tid; i < nch * rows; i += kWideEpiThreads) dst[i] = src[i];
        return;
      }
      unsigned char* d0 = nullptr;                   // (the input dump ACT[0] is a bulk store issued at the stage's start)
      for (int j = 0; j < 2; ++j) {
        const RowCtx rc = rowctx(j, tile);
        for (int c8 = ch; c8 < nch0; c8 += 2) {
          uint4 q = make_uint4(0, 0, 0, 0);
          if (rc.valid) {
            size_t base = ((size_t)rc.gw * T + rc.t) * n_in;
            if constexpr (MODE == 0 || VIEW) {
              if (p.wv.win_start) {                  // window view: the source row in the frame stream
                const long long f = window_src_row(p.wv, rc.gw, rc.t);
                if (f < 0) {                         // a zero row: no keypoints, the pos-emb channel as in a padded window
                  if (pe && c8 == 0) q.x = pack_bf16x2(__fdiv_rn((float)rc.t, (float)g.pe_len), 0.0f);
                  *reinterpret_cast<uint4*>(A + (size_t)c8 * CH + (size_t)rc.row * 16) = q;
                  continue;
                }
                base = (size_t)f * n_in;
              }
            }
            if (vec_in && c8 * 8 < n_in) {
              if (p.x_dtype == B2H_DT_F32) {
                const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.x) + base) + 2 * c8;
                const float4 lo = __ldg(src), hi = __ldg(src + 1);
                q.x = pack_bf16x2(lo.x, lo.y); q.y = pack_bf16x2(lo.z, lo.w);
                q.z = pack_bf16x2(hi.x, hi.y); q.w = pack_bf16x2(hi.z, hi.w);
              } else {
                q = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.x) + base) + c8);
              }
            } else if (!vec_in) {
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int cc = c8 * 8 + e;          // channel in the conv1 input (pos-emb row first)
                float val = 0.0f;
                if (pe && cc == 0) val = __fdiv_rn((float)rc.t, (float)g.pe_len);             // HandPoseModels.py:70-82
                else if (cc - pe < n_in && cc - pe >= 0)
                  val = (p.x_dtype == B2H_DT_F32) ? __ldg(reinterpret_cast<const float*>(p.x) + base + (cc - pe))
                                                  : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.x)[base + (cc - pe)]);
                v[e] = val;
              }
              q.x = pack_bf16x2(v[0], v[1]); q.y = pack_bf16x2(v[2], v[3]);
              q.z = pack_bf16x2(v[4], v[5]); q.w = pack_bf16x2(v[6], v[7]);
            }
          }
          *reinterpret_cast<uint4*>(A + (size_t)c8 * CH + (size_t)rc.row * 16) = q;
          if (d0) *reinterpret_cast<uint4*>(d0 + (size_t)c8 * CH + (size_t)rc.row * 16) = q;
        }
      }
    };
    auto publish = [&]() {                    // my smem writes -> async proxy, my TMEM reads are done
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(&act_ready);
    };
    auto pack8 = [&](const float* f) {
      uint4 q;
      q.x = pack_bf16x2(f[0], f[1]); q.y = pack_bf16x2(f[2], f[3]);
      q.z = pack_bf16x2(f[4], f[5]); q.w = pack_bf16x2(f[6], f[7]);
      return q;
    };

    stage_inputs(blockIdx.x);
    publish();
    uint32_t acc_phase = 0;
    int en = 64;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      for (int l = 0; l < NL; ++l) {
        const int N = p.st[l].N;
        const int layer = p.st[l].layer;      // model layer this stage belongs to (forward: l; backward: 3, 2, 1)
        // MODE 2: the ReLU mask of this stage (saved input of `layer` > 0) is fetched from the scratch dump and compressed
        // to bits WHILE the stage's MMAs run -- inside the epilogue loop the 32 dependent global loads per thread cost more
        // than the accumulator read-out itself.  bit (32 it + 8 i + q) = channel 32 ch + 64 it + 8 i + q of this thread's row.
        uint32_t mb0[4] = {0u, 0u, 0u, 0u}, mb1[4] = {0u, 0u, 0u, 0u};
        if (MODE == 2) {
          const RowCtx rc0 = rowctx(0, tile), rc1 = rowctx(1, tile);
          const unsigned char* am = dump(tile, p.act_off[layer]);
          auto pos8 = [](const uint4& a) {      // 8 bf16 -> 8 bits (value > 0)
            const uint32_t w[4] = {a.x, a.y, a.z, a.w};
            uint32_t b = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const uint32_t lo = w[e] & 0xFFFFu, hi = w[e] >> 16;
              b |= (uint32_t)(((lo & 0x8000u) == 0u) && ((lo & 0x7FFFu) != 0u)) << (2 * e);
              b |= (uint32_t)(((hi & 0x8000u) == 0u) && ((hi & 0x7FFFu) != 0u)) << (2 * e + 1);
            }
            return b;
          };
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int c0 = 32 * ch + 64 * it;
            if (c0 < N) {
              uint4 a0[4], a1[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const bool in = c0 + 8 * i < N;
                const size_t o0 = (size_t)((c0 >> 3) + i) * CH + (size_t)rc0.row * 16, o1 = (size_t)((c0 >> 3) + i) * CH + (size_t)rc1.row * 16;
                a0[i] = in ? __ldg(reinterpret_cast<const uint4*>(am + o0)) : make_uint4(0, 0, 0, 0);
                a1[i] = in ? __ldg(reinterpret_cast<const uint4*>(am + o1)) : make_uint4(0, 0, 0, 0);
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) { mb0[it] |= pos8(a0[i]) << (8 * i); mb1[it] |= pos8(a1[i]) << (8 * i); }
            }
          }
          if (!rc0.valid) { mb0[0] = mb0[1] = mb0[2] = mb0[3] = 0u; }
          if (!rc1.valid) { mb1[0] = mb1[1] = mb1[2] = mb1[3] = 0u; }
        }
        if (!mbar_wait(&acc_full, acc_phase, 63 + l)) return;
        acc_phase ^= 1;
        tc_fence_after();
        if (p.dbg && blockIdx.x == 0 && tid == 0 && en < 124) p.dbg[en++] = clock64();   // accumulators complete
        if (MODE == 2 || l < 3) {
          // both 128-row accumulators' chunks are fetched before one wait: two TMEM loads in flight per thread
          const RowCtx rc0 = rowctx(0, tile), rc1 = rowctx(1, tile);
          const uint32_t taddr = tbase + lane_addr;
          // MODE 1: a_{l+1} = input of layer l+1 -> ACT[l+1];  MODE 2: dZ_{layer-1} -> DZ[layer-1], masked by the saved
          // input of `layer` (= a_layer = relu output of layer-1)
          // MODE 2, last stage: dZ_0 has no later stage whose start would dump it -> stored by these threads
          unsigned char* dd = (MODE == 2 && l == NL - 1) ? dump(tile, p.dz_off[layer - 1]) : nullptr;
          if (dd) zero_halo(dd, N / 8);
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int c0 = 32 * ch + 64 * it;
            if (c0 >= N) break;
            uint32_t v0[32], v1[32];
            tmem_ld32(taddr + c0, v0);
            tmem_ld32(taddr + 256 + c0, v1);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (c0 + 8 * i >= N) continue;          // N is a multiple of 16: never write a chunk past the layer's columns
              float f0[8], f1[8];
              if (MODE != 2) {
                const float4 b0 = *reinterpret_cast<const float4*>(&bias_s[l][c0 + 8 * i]);
                const float4 b1 = *reinterpret_cast<const float4*>(&bias_s[l][c0 + 8 * i + 4]);
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                  f0[q] = rc0.valid ? fmaxf(__uint_as_float(v0[8 * i + q]) + bb[q], 0.0f) : 0.0f;
                  f1[q] = rc1.valid ? fmaxf(__uint_as_float(v1[8 * i + q]) + bb[q], 0.0f) : 0.0f;
                }
              } else {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                  f0[q] = ((mb0[it] >> (8 * i + q)) & 1u) ? __uint_as_float(v0[8 * i + q]) : 0.0f;
                  f1[q] = ((mb1[it] >> (8 * i + q)) & 1u) ? __uint_as_float(v1[8 * i + q]) : 0.0f;
                }
              }
              const uint4 q0 = pack8(f0), q1 = pack8(f1);
              const size_t o0 = (size_t)((c0 >> 3) + i) * CH + (size_t)rc0.row * 16, o1 = (size_t)((c0 >> 3) + i) * CH + (size_t)rc1.row * 16;
              // MODE 2, last stage: dZ_0 goes to the dump only.  The buffer already belongs to the CTA's next tile: epilogue
              // threads that finish first copy that tile's dZ_4 into it (stage_inputs below, with no barrier in between),
              // and a late store of dZ_0 here would overwrite it.
              unsigned char* out = dd ? dd : A;
              *reinterpret_cast<uint4*>(out + o0) = q0;
              *reinterpret_cast<uint4*>(out + o1) = q1;
            }
          }
        } else if (MODE == 0) {
          for (int j = 0; j < 2; ++j) {
            const RowCtx rc = rowctx(j, tile);
            const uint32_t taddr = tbase + lane_addr + 256 * j;
            // layer 4: prediction rows (+ mask_output utils.py:309-312, de-normalisation) straight to global memory
            int len = T;
            if (rc.valid && p.lengths) { len = p.lengths[rc.gw]; len = len < 0 ? 0 : (len > T ? T : len); }
            float* yrow = rc.valid ? p.y + ((size_t)rc.gw * T + rc.t) * B2H_COUT : nullptr;
            const bool masked = p.apply_mask && (rc.t >= len);
            for (int c0 = 16 * ch; c0 < N; c0 += 32) {
              uint32_t v[16];
              tmem_ld16(taddr + c0, v);
              tmem_ld_wait();
#pragma unroll
              for (int q = 0; q < 16; q += 2) {
                const int c = c0 + q;
                if (yrow && c < B2H_COUT) {
                  float a = __uint_as_float(v[q]) + bias_s[3][c];
                  float b = __uint_as_float(v[q + 1]) + bias_s[3][c + 1];
                  if (masked) { a = 0.0f; b = 0.0f; }
                  else if (p.out_scale != 1.0f) { a *= p.out_scale; b *= p.out_scale; }
                  *reinterpret_cast<float2*>(yrow + c) = make_float2(a, b);
                }
              }
            }
          }
        } else {
          // MODE 1, layer 4: masked prediction, criterion term and d(loss)/d(pred) -> DZ[3] (bf16), optional prediction rows.
          // L1 is the confidence-weighted form with s = 1 (a*1 - t*1 == a - t exactly).   utils.py:422-426 / :447-450
          unsigned char* dd = dump(tile, p.dz_off[3]);
          zero_halo(dd, N / 8);
          for (int j = 0; j < 2; ++j) {
            const RowCtx rc = rowctx(j, tile);
            const uint32_t taddr = tbase + lane_addr + 256 * j;
            int len = T;
            if (rc.valid && p.lengths) { len = p.lengths[rc.gw]; len = len < 0 ? 0 : (len > T ? T : len); }
            const bool live = rc.valid && (rc.t < len);
            const float n_el = (float)len * (float)B2H_COUT;
            const float scale = !live ? 0.f : ((p.loss_kind == B2H_LOSS_L1) ? (1.0f / (float)p.B) / n_el : 1.0f / n_el);
            const size_t ro = rc.valid ? ((size_t)rc.gw * T + rc.t) : 0;
            size_t tro = ro;                         // row of the target / confidences: a stream row for a window view
            bool zrow = false;                       // ... or a zero row (its target and confidences read as zeros)
            if (VIEW && rc.valid) {
              const long long f = window_src_row(p.wv, rc.gw, rc.t);
              zrow = f < 0;
              tro = zrow ? 0 : (size_t)f;
            }
            const float* tg = p.train_mode == 1 ? p.target + tro * B2H_COUT : p.d_y + ro * B2H_COUT;
            const float* cf = (p.conf && p.loss_kind == B2H_LOSS_CONFL1) ? p.conf + tro * (B2H_COUT / 2) : nullptr;
            float* yrow = (rc.valid && p.y) ? p.y + ro * B2H_COUT : nullptr;
            float sum = 0.f;
            for (int c0 = 16 * ch; c0 < N; c0 += 32) {
              uint32_t v[16];
              tmem_ld16(taddr + c0, v);
              tmem_ld_wait();
              float gq[16];
#pragma unroll
              for (int q = 0; q < 16; q += 2) {
                const int c = c0 + q;
                float2 tv = make_float2(0.f, 0.f);
                float sv = 1.0f;
                const bool on = live && c < B2H_COUT;
                if (on) {
                  tv = __ldg(reinterpret_cast<const float2*>(tg + c));
                  if (cf) sv = __ldg(cf + (c >> 1));
                  if (VIEW && zrow) { tv = make_float2(0.f, 0.f); sv = cf ? 0.f : 1.0f; }
                }
                const float a0 = on ? __uint_as_float(v[q]) + bias_s[3][c < 255 ? c : 255] : 0.0f;
                const float a1 = on ? __uint_as_float(v[q + 1]) + bias_s[3][c < 254 ? c + 1 : 255] : 0.0f;
                if (p.train_mode == 1) {
                  const float d0 = __fsub_rn(__fmul_rn(a0, sv), __fmul_rn(tv.x, sv));
                  const float d1 = __fsub_rn(__fmul_rn(a1, sv), __fmul_rn(tv.y, sv));
                  sum += on ? fabsf(d0) : 0.0f;
                  sum += on ? fabsf(d1) : 0.0f;
                  const float sc = sv * scale;
                  gq[q] = on ? (d0 > 0.f ? sc : (d0 < 0.f ? -sc : 0.f)) : 0.0f;
                  gq[q + 1] = on ? (d1 > 0.f ? sc : (d1 < 0.f ? -sc : 0.f)) : 0.0f;
                } else {                               // backward of a given d_y: the loaded value IS the gradient
                  gq[q] = on ? tv.x : 0.0f;
                  gq[q + 1] = on ? tv.y : 0.0f;
                }
                if (yrow && c < B2H_COUT) *reinterpret_cast<float2*>(yrow + c) = make_float2(a0, a1);
              }
              *reinterpret_cast<uint4*>(dd + (size_t)(c0 >> 3) * CH + (size_t)rc.row * 16) = pack8(gq);
              *reinterpret_cast<uint4*>(dd + (size_t)((c0 >> 3) + 1) * CH + (size_t)rc.row * 16) = pack8(gq + 8);
            }
            // per-sample mean = sum_{t<len} |d| / (len*42)  (utils.py:426 / :450)
            if (p.train_mode == 1 && live) loss_run += sum / n_el;
          }
        }
        if (l == NL - 1) stage_inputs(tile + gridDim.x);   // the buffer is dead after the last stage's MMAs: next tile's rows go in
        publish();
        if (p.dbg && blockIdx.x == 0 && tid == 0 && en < 124) p.dbg[en++] = clock64();   // epilogue done
      }
    }
    if (MODE == 1) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) loss_run += __shfl_xor_sync(0xffffffffu, loss_run, o);
      if (lane == 0) loss_w[warp] = loss_run;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (MODE == 1 && tid == 0 && p.loss_partials) {
    const float s = ((loss_w[0] + loss_w[1]) + (loss_w[2] + loss_w[3])) + ((loss_w[4] + loss_w[5]) + (loss_w[6] + loss_w[7]));
    p.loss_partials[blockIdx.x] = (p.loss_kind == B2H_LOSS_L1) ? s / (float)p.B : s;
  }
  if (warp == 0) tmem_dealloc(tbase, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// Weight gradients of the wide training path: split-K GEMMs over the scratch dumps.
//   dW_l[k][co][ci] = sum_r dZ_l[r][co] * in_l[r+k-2][ci],   db_l[co] = sum_r dZ_l[r][co]      (r over all rows of all tiles)
// Both operands are the dumps read MN-major (K = rows, 16 per MMA): A = dZ_l (M = 128 output channels, or 64 for conv4),
// B = in_l shifted by the tap (N <= 64 input channels), accumulators = 5 taps x N columns (+ 8 for the bias gradient against
// a ones column) in TMEM.  Work item = (layer, co block, ci block); every item is split over `ksplit` CTAs by tile range;
// each CTA writes its accumulators once into its slice of the partials workspace in the gradient-partial slot layout
// (b2h_common.cuh gp_*), which the Adam / reduce kernels sum in fixed order (deterministic).
// Pipeline: one producer thread streams the tile's A / B pieces (contiguous runs of chunks) into a 2-stage ring with TMA
// tensor-map loads (the scratch viewed as rows of 128 B, box = 4 chunks = 132 rows; 1-D bulk copies top out at
// ~23 B/cycle/SM, below the 32 B/cycle the MMAs consume); one thread issues the MMAs; 4 warps read the accumulators out.
struct WgradItem { int l, m0, M, n0, N, with_bias; };
constexpr int kWgMaxItems = 48;
struct WgradArgs {
  const unsigned char* scratch;
  long long tile_bytes, act_off[4], dz_off[4];
  int n_tiles, n_items, ksplit;
  float* partials;          // [ksplit][gp_total]
  Geo geo;
  WgradItem items[kWgMaxItems];
};
constexpr int kWgThreads = 192;           // warp 0: producer, warp 1: MMA issuer, warps 2..5: read-out (TMEM lane quadrants 2,3,0,1)
constexpr int kWgChunkB = kWideRows * 16; // bytes of one 8-channel chunk of a dump
constexpr int kWgABytes = 16 * kWgChunkB; // A piece: up to 16 chunks (M = 128)
constexpr int kWgBBytes = 8 * kWgChunkB;  // B piece: up to 8 chunks (N = 64)
constexpr int kWgStageBytes = kWgABytes + kWgBBytes;
constexpr int kWgBiasCol = 5 * 64;
constexpr int kWgBoxChunks = 4;           // chunks per TMA box
constexpr int kWgBoxRows = kWgBoxChunks * kWgChunkB / 128;   // 132 rows of 128 B
constexpr int kWgBoxBytes = kWgBoxChunks * kWgChunkB;

__global__ void __launch_bounds__(kWgThreads, 1) conv_tc_wide_wgrad_kernel(WgradArgs p, const __grid_constant__ CUtensorMap smap) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full_bar[2], empty_bar[2], done_bar;
  __shared__ uint32_t tmem_slot;
  const Geo& g = p.geo;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int item_id = blockIdx.x % p.n_items, split = blockIdx.x / p.n_items;
  const WgradItem it = p.items[item_id];
  const int per = (p.n_tiles + p.ksplit - 1) / p.ksplit;
  const int t0 = split * per, t1 = min(p.n_tiles, t0 + per);
  unsigned char* ONES = smem + 2 * kWgStageBytes;
  // ones column (B operand of the bias-gradient GEMM): element 0 of every row = 1.0 (dZ is zero on non-frame rows); a
  // second, zero chunk behind it because an M = 128 MMA needs N >= 16
  for (int i = tid; i < 2 * kWideRows; i += kWgThreads)
    *reinterpret_cast<uint4*>(ONES + (size_t)i * 16) = make_uint4(i < kWideRows ? 0x00003F80u : 0u, 0, 0, 0);
  // chunks of the A piece beyond the layer's channels (M = 64 reads 8 chunks, conv4 has 6) must hold finite values: zero them once
  {
    const int a_chunks = min(it.M / 8, g.np_[it.l] / 8 - it.m0 / 8);
    for (int s = 0; s < 2; ++s)
      for (int i = tid; i < (16 - a_chunks) * kWideRows; i += kWgThreads)
        *reinterpret_cast<uint4*>(smem + (size_t)s * kWgStageBytes + (size_t)a_chunks * kWgChunkB + (size_t)i * 16) = make_uint4(0, 0, 0, 0);
    const int b_chunks = min(it.N / 8, g.kp[it.l] / 8 - it.n0 / 8);
    for (int s = 0; s < 2; ++s)
      for (int i = tid; i < (8 - b_chunks) * kWideRows; i += kWgThreads)
        *reinterpret_cast<uint4*>(smem + (size_t)s * kWgStageBytes + kWgABytes + (size_t)b_chunks * kWgChunkB + (size_t)i * 16) = make_uint4(0, 0, 0, 0);
  }
  if (warp == 0) tmem_alloc(&tmem_slot, 512);
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&done_bar, 1);
    fence_barrier_init();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;
  const int a_chunks = min(it.M / 8, g.np_[it.l] / 8 - it.m0 / 8);
  const int b_chunks = min(it.N / 8, g.kp[it.l] / 8 - it.n0 / 8);
  const int a_boxes = (a_chunks + kWgBoxChunks - 1) / kWgBoxChunks, b_boxes = (b_chunks + kWgBoxChunks - 1) / kWgBoxChunks;

  if (warp == 0) {
    if (elect_one()) {
      uint32_t ph = 1;
      int s = 0;
      const uint32_t full0 = smem_u32(&full_bar[0]);
      for (int tile = t0; tile < t1; ++tile) {
        if (!mbar_wait(&empty_bar[s], ph, 70)) break;
        // 128-byte row of the tile's A / B piece in the scratch tensor (every offset is a multiple of one chunk = 33 rows)
        const long long base = (long long)tile * p.tile_bytes;
        const int arow = (int)((base + p.dz_off[it.l] + (long long)(it.m0 / 8) * kWgChunkB) >> 7);
        const int brow = (int)((base + p.act_off[it.l] + (long long)(it.n0 / 8) * kWgChunkB) >> 7);
        const uint32_t st = smem_u32(smem + (size_t)s * kWgStageBytes);
        expect_tx_addr(full0 + s * 8, (uint32_t)(a_boxes + b_boxes) * kWgBoxBytes);      // a box past the tensor end is zero-filled, still counted
        for (int b = 0; b < a_boxes; ++b) tma_load_2d_addr(st + b * kWgBoxBytes, &smap, 0, arow + b * kWgBoxRows, full0 + s * 8);
        for (int b = 0; b < b_boxes; ++b) tma_load_2d_addr(st + kWgABytes + b * kWgBoxBytes, &smap, 0, brow + b * kWgBoxRows, full0 + s * 8);
        if (++s == 2) { s = 0; ph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {
      uint32_t ph = 0;
      int s = 0;
      const uint32_t hi_mn = desc_hi((uint32_t)kWgChunkB);           // MN-major: SBO = chunk stride, LBO = 128 B (8 rows)
      const uint32_t idw = make_idesc_bf16(it.M, it.N, 1, 1), idb = make_idesc_bf16(it.M, it.M == 128 ? 16 : 8, 1, 1);
      const uint32_t o_lo = desc_lo(smem_u32(ONES), 128);
      uint32_t first = 0;
      for (int tile = t0; tile < t1; ++tile) {
        if (!mbar_wait(&full_bar[s], ph, 71)) break;
        const uint32_t a_lo = desc_lo(smem_u32(smem + (size_t)s * kWgStageBytes), 128);
        const uint32_t b_lo = desc_lo(smem_u32(smem + (size_t)s * kWgStageBytes + kWgABytes), 128);
        for (int ks = 0; ks < 16; ++ks) {
          const uint32_t r0 = 2 + 16 * ks;                             // output rows 2 + 16 ks .. (16-B units)
          const uint64_t ad = desc64(a_lo + r0, hi_mn);
#pragma unroll
          for (int k = 0; k < B2H_KW; ++k) umma_bf16(tbase + k * 64, ad, desc64(b_lo + r0 + k - 2, hi_mn), idw, first);
          if (it.with_bias) umma_bf16(tbase + kWgBiasCol, ad, desc64(o_lo + r0, hi_mn), idb, first);
          first = 1;
        }
        umma_commit(&empty_bar[s]);                                    // stage reusable once these MMAs have read it
        if (++s == 2) { s = 0; ph ^= 1; }
      }
      umma_commit(&done_bar);
    }
    __syncwarp();
  } else {
    // ===== read-out: TMEM lane quadrant = warp & 3; lane -> output channel =====
    mbar_wait(&done_bar, 0, 72);
    tc_fence_after();
    const int q = warp & 3;
    const int l = it.l;
    const int co = it.M == 128 ? it.m0 + q * 32 + lane : it.m0 + q * 16 + (lane & 15);     // M = 64: rows live in lanes 32q + i, i < 16
    const bool mine = (it.M == 128 || lane < 16) && co < g.cout[l] && t1 > t0;
    const bool zero = t1 <= t0;                                                          // a split without tiles contributes zeros
    float* part = p.partials + (size_t)split * gp_total(g) + gp_layer_off(g, l);
    float4* lp4 = reinterpret_cast<float4*>(part);
    const int q4 = g.kp[l] >> 2, cout_l = g.cout[l];
    const uint32_t taddr = tbase + ((uint32_t)(q * 32) << 16);
    const bool row_ok = (it.M == 128 || lane < 16) && co < g.cout[l];
    for (int k = 0; k < B2H_KW; ++k)
      for (int c0 = 0; c0 < it.N; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(taddr + k * 64 + c0, v);
        tmem_ld_wait();
        if (row_ok) {
          float4* dst = lp4 + ((size_t)k * q4 + ((it.n0 + c0) >> 2)) * cout_l + co;
#pragma unroll
          for (int qq = 0; qq < 4; ++qq)
            if (it.n0 + c0 + 4 * qq < g.kp[l])
              dst[(size_t)qq * cout_l] = zero ? make_float4(0.f, 0.f, 0.f, 0.f)
                                              : make_float4(__uint_as_float(v[4 * qq]), __uint_as_float(v[4 * qq + 1]),
                                                            __uint_as_float(v[4 * qq + 2]), __uint_as_float(v[4 * qq + 3]));
        }
      }
    if (it.with_bias) {
      uint32_t vb[16];
      tmem_ld16(taddr + kWgBiasCol, vb);
      tmem_ld_wait();
      if (row_ok) part[B2H_KW * cout_l * g.kp[l] + co] = zero ? 0.0f : __uint_as_float(vb[0]);
    }
    (void)mine;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, 512);
}

// ---- host side ----
static int wide_wgrad_items(const Geo& g, WgradItem* items) {
  int n = 0;
  for (int l = 0; l < 4; ++l) {
    const int M = g.np_[l] <= 64 ? 64 : 128;
    for (int m0 = 0; m0 < g.np_[l]; m0 += M)
      for (int n0 = 0; n0 < g.kp[l]; n0 += 64) {
        if (n >= kWgMaxItems) return -1;
        const int N = g.kp[l] - n0 < 64 ? g.kp[l] - n0 : 64;
        items[n++] = WgradItem{l, m0, M, n0, N, n0 == 0 ? 1 : 0};
      }
  }
  return n;
}

// 220 KB hold the activation buffer and a ring of 3..16 weight stages; a tile holds gh whole windows; training splits
// the weight-gradient GEMMs K-wise over the tiles so that items x ksplit CTAs about fill the SMs.
WidePlan plan_wide(const Geo& g, int B, int T) {
  WidePlan p{};
  if (T < 1 || T > 256 || g.C > 256 || g.cin[0] > 64) return p;
  int kmax = g.kp[0];
  for (int l = 1; l < 4; ++l) kmax = kmax > g.kp[l] ? kmax : g.kp[l];
  for (int l = 0; l < 4; ++l) kmax = kmax > g.np_[l] ? kmax : g.np_[l];
  p.a_bytes = (kmax / 8) * kWideRows * 16;
  int S = (int)(((size_t)220 * 1024 - p.a_bytes) / kWideStage);
  if (S > kWideMaxStages) S = kWideMaxStages;
  p.ok = S >= 3;
  p.nstage = S;
  p.smem = (size_t)p.a_bytes + (size_t)S * kWideStage;
  p.gh = 258 / (T + 2);
  p.n_tiles = (B + p.gh - 1) / p.gh;
  const int sms = num_sms();
  p.grid = sms < p.n_tiles ? sms : p.n_tiles;
  p.n_loss = p.grid;
  p.scratch_bytes = (int64_t)p.n_tiles * wide_scratch(g).tile_bytes;
  WgradItem items[kWgMaxItems];
  const int n = wide_wgrad_items(g, items);
  p.ksplit = n > 0 ? sms / n : 1;
  if (p.ksplit < 1) p.ksplit = 1;
  if (p.ksplit > p.n_tiles) p.ksplit = p.n_tiles;
  return p;
}

// tensor map over a run of packed UMMA weight sections viewed as rows of 64 bf16 (128 B), box = 128 rows (one ring stage)
static int wide_weight_map(const char* base, int64_t bytes, CUtensorMap* out, int box_rows = kWideBoxRows) {
  typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeTiledFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || !fn) { cudaGetLastError(); set_error("cuTensorMapEncodeTiled entry point unavailable"); return B2H_ECUDA; }
    encode = (EncodeTiledFn)fn;
  }
  const cuuint64_t gdim[2] = {64, (cuuint64_t)(bytes >> 7)};
  const cuuint64_t gstride[1] = {128};
  const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<char*>(base), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return B2H_ECUDA; }
  return B2H_OK;
}

// The forward's and the training forward's arguments (mode 0: the training fields stay zero in `a`), with the four
// forward conv stages.
static WideArgs wide_args(const ConvArgs& a, const WidePlan& plan) {
  const Geo& g = a.geo;
  WideArgs p{};
  p.x = a.x; p.x_dtype = a.x_dtype; p.params = a.params; p.packed = a.packed; p.lengths = a.lengths; p.y = a.y;
  p.apply_mask = a.apply_mask; p.out_scale = a.out_scale;
  p.target = a.target; p.conf = a.conf; p.d_y = a.d_y; p.loss_kind = a.loss_kind; p.train_mode = a.mode;
  p.loss_partials = a.loss_partials; p.step_dev = a.step_dev; p.epoch_dev = a.epoch_dev;
  p.wv = a.wv;
  p.B = a.B; p.T = a.T; p.geo = g;
  p.dbg = g_dbg_timing;
  p.gh = plan.gh; p.n_tiles = plan.n_tiles; p.a_bytes = plan.a_bytes; p.nstage = plan.nstage;
  const WideScratch ws = wide_scratch(g);
  p.tile_bytes = ws.tile_bytes;
  for (int l = 0; l < 4; ++l) { p.act_off[l] = ws.act_off[l]; p.dz_off[l] = ws.dz_off[l]; }
  p.n_stages = 4;
  for (int l = 0; l < 4; ++l) { p.st[l].KS = g.kp[l] >> 4; p.st[l].N = g.np_[l]; p.st[l].row0 = (int)((g.tf_off[l] - g.tf_off[0]) >> 7); p.st[l].layer = l; }
  return p;
}

int launch_tc_wide_fwd(const ConvArgs& a, const WidePlan& plan, cudaStream_t stream) {
  const Geo& g = a.geo;
  const WideArgs p = wide_args(a, plan);
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_tc_wide_kernel<0>), plan.smem)) return rc;
  CUtensorMap wmap;
  if (int rc = wide_weight_map(a.packed + g.tf_off[0], g.td_off[0] - g.tf_off[0], &wmap)) return rc;
  conv_tc_wide_kernel<0><<<plan.grid, kWideThreads, plan.smem, stream>>>(p, wmap);
  count_launch();
  return check_launch("conv_tc_wide_kernel<fwd>");
}

// ---- wide training: forward+criterion (saves layer inputs), dgrad chain, split-K wgrad; the caller reduces + applies Adam ----
int launch_tc_wide_train(const ConvArgs& a, const WidePlan& plan, unsigned char* scratch, cudaStream_t stream) {
  const Geo& g = a.geo;
  WideArgs p = wide_args(a, plan);
  p.scratch = scratch;
  const size_t smem = plan.smem;
  const int grid = plan.grid;
  // ---- 1. forward + criterion ----
  auto* fwd = p.wv.win_start ? conv_tc_wide_kernel<1, true> : conv_tc_wide_kernel<1>;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fwd), smem)) return rc;
  CUtensorMap fmap, bmap;
  if (int rc = wide_weight_map(a.packed + g.tf_off[0], g.td_off[0] - g.tf_off[0], &fmap)) return rc;
  fwd<<<grid, kWideThreads, smem, stream>>>(p, fmap);
  count_launch();
  if (int rc = check_launch("conv_tc_wide_kernel<train fwd>")) return rc;
  // ---- 2. dgrad chain: layers 4, 3, 2 with the transposed blocks (td sections are contiguous from td_off[1]) ----
  if (int rc = wide_weight_map(a.packed + g.td_off[1], g.tfl_off[0] - g.td_off[1], &bmap)) return rc;
  p.n_stages = 3;
  for (int j = 0; j < 3; ++j) {
    const int l = 3 - j;
    p.st[j].KS = g.np_[l] >> 4; p.st[j].N = g.kp[l]; p.st[j].row0 = (int)((g.td_off[l] - g.td_off[1]) >> 7); p.st[j].layer = l;
  }
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_tc_wide_kernel<2>), smem)) return rc;
  conv_tc_wide_kernel<2><<<grid, kWideThreads, smem, stream>>>(p, bmap);
  count_launch();
  if (int rc = check_launch("conv_tc_wide_kernel<dgrad>")) return rc;
  // ---- 3. weight / bias gradients: split-K GEMMs over the dumps ----
  WgradArgs w{};
  w.scratch = scratch; w.tile_bytes = p.tile_bytes;
  for (int l = 0; l < 4; ++l) { w.act_off[l] = p.act_off[l]; w.dz_off[l] = p.dz_off[l]; }
  w.n_tiles = p.n_tiles; w.partials = a.partials; w.geo = g;
  w.n_items = wide_wgrad_items(g, w.items);
  if (w.n_items <= 0) { set_error("wide wgrad: too many work items"); return B2H_ESHAPE; }
  w.ksplit = plan.ksplit;
  const size_t wsmem = (size_t)2 * kWgStageBytes + 2 * kWgChunkB;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_tc_wide_wgrad_kernel), wsmem)) return rc;
  CUtensorMap smap;
  if (int rc = wide_weight_map(reinterpret_cast<const char*>(scratch), (int64_t)p.n_tiles * p.tile_bytes, &smap, kWgBoxRows)) return rc;
  conv_tc_wide_wgrad_kernel<<<w.n_items * w.ksplit, kWgThreads, wsmem, stream>>>(w, smap);
  count_launch();
  return check_launch("conv_tc_wide_wgrad_kernel");
}

}  // namespace b2h
