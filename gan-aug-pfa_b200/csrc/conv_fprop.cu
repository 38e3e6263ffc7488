// Implicit-GEMM convolution engine ("fprop-like" contraction) for sm_100a.
//
//   D[pixel, co] = sum_k A[pixel, k] * B[co, k]
//
// A is never materialised: a tile of 128 output-grid points (BW x BH x BNI, all powers of two) is
// fetched per filter tap and per 64-channel chunk straight from the NHWC bf16 activation tensor
// by ONE 4-D tiled TMA box (traversal stride = conv stride, out-of-bounds = zero padding) into a
// 128-byte-swizzled K-major shared-memory tile that tcgen05.mma consumes through a shared-memory
// matrix descriptor.  B (packed weights, K-major) comes through a second TMA box.  Accumulators
// live in TMEM (two 256-column buffers, so the epilogue of tile i overlaps the main loop of tile
// i+1).  Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM allocator), warps 2..5 =
// epilogue (tcgen05.ld -> bias -> BatchNorm partial statistics -> activation(s) -> bf16 stores).
//
// The same kernel serves Conv2d forward, Conv2d dgrad (stride 1: flipped taps; stride 2: four
// output-parity phases of 2x2 taps), ConvTranspose2d forward (the same four phases) and
// ConvTranspose2d dgrad (a strided gather) — see gap_b200.h.
#include "common.h"
#include "ptx.cuh"
#include "mma_sync.cuh"

namespace gap {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KiB
constexpr int kEpiWarps = 8;   // two warps per TMEM lane quarter: one warp per scheduler is latency-bound in the epilogue
constexpr int kProducer2Warp = 2 + kEpiWarps;   // second TMA producer warp (takes the odd pipeline iterations)
constexpr int kFpropThreads = 64 + 32 * kEpiWarps + 32;
constexpr int kMaxStages = 8;
constexpr int kAccStride = 256;  // TMEM columns between the two accumulator buffers
constexpr int kTmemCols = 512;
constexpr int kStatsBytes = 4 * 256 * 2 * 8;  // per-epilogue-warp fp64 partial sums
constexpr int kBarrierBytes = 256;
constexpr int kParamBytes = 2 * 256 * 4;  // per-N-tile scale / shift of the backward-fused epilogue
constexpr int kColStageBytes = kEpiWarps * 1024;  // per-epilogue-warp 32x16 bf16 tile for the column sums
constexpr int kSmemBudget = 227 * 1024;

struct alignas(64) FpropParams {
  CUtensorMap tmA[2];
  CUtensorMap tmB;
  int src_chunks[2];
  int n_img, gh, gw;
  int n_phase, taps_h, taps_w, in_stride;
  int in_off_h[2], in_off_w[2];
  int out_stride;
  int log_bw, log_bh;
  int tiles_w, tiles_h, tiles_n;
  int n_tiles, block_n;
  int n_out, OH, OW;
  __nv_bfloat16* out;
  long long out_ld;
  int act;
  __nv_bfloat16* out2;
  long long out2_ld;
  int act2;
  const float* bias;
  const float* scale;   // per-channel multiplier applied before the bias (eval-mode BatchNorm folded into the epilogue)
  double* stats;
  int num_stages;
  uint32_t idesc;
  int total_tiles;
  int k_iters;
  int mt;          // M tiles (128 rows each) per CTA work item: they share every B tile fetched from L2
  int sm_tiles;    // work items along M per phase = ceil(m_tiles_pp / mt)
  int m_tiles_pp;  // M tiles per phase
  int acc_stages;  // TMEM accumulator buffers (2 when mt*block_n <= 256, else 1)
  int vec_ok;  // 1: outputs 16-byte aligned per pixel (128-bit stores); 2: 32-byte aligned (256-bit)
  int out_f32;  // `out` is fp32 (scalar stores; used for the 1-channel logits)
  int fast_store;  // slope-type activations and 32-byte-aligned bf16 outputs: vector epilogue
  float slope1, slope2;  // negative-side slope of act / act2 (1 identity, 0.2 LeakyReLU, 0 ReLU)
  // backward-fused epilogue (kEpi = 1): activation (+BatchNorm) backward applied to output channels >= bwd_c0
  const __nv_bfloat16* bwd_y;
  long long bwd_y_ld;
  const float* bwd_scale;
  const float* bwd_shift;
  const __nv_bfloat16* bwd_g2;
  long long bwd_g2_ld;
  float bwd_slope;
  int bwd_c0;
  int bwd_ld32;   // y / g2 rows allow 256-bit loads
  int skip;  // bring-up ablation: 1 no global stores, 2 no y / g2 loads, 4 no statistics
  int accum;  // kEpi = 2: out[pix][c] = act(v) + out[pix][c] (a gradient with several contributors)
  // Halo mode: the taps of one kernel column that differ only by whole input rows (th = g + in_stride*i) share ONE
  // A tile of BH + halo_taps - 1 rows; tap i reads it through a descriptor shifted by i*BW rows (BW % 8 == 0, so the
  // shift is a whole number of 1024-byte swizzle atoms).  Cuts the A-operand TMA traffic of small-N layers.
  int halo;            // 0 / 1
  int halo_taps;       // taps per group (taps_h / in_stride)
  int halo_groups;     // in_stride
  int a_tile_bytes;    // bytes of one A tile in shared memory (16 KiB, or the halo tile rounded up to 1 KiB)
  int a_load_bytes;    // bytes one A TMA load delivers
  int b_per_stage;     // B tiles per pipeline stage (1, or halo_taps)
  int chunks_tot;      // 64-channel chunks over both sources
  // CTA-pair mode (kPair, see ptx.cuh "CTA pairs"): a cluster of two CTAs works on ONE work item of 2*mt M tiles; CTA
  // rank r owns M tiles (2*sm + r)*mt .. +mt and stages rows [r*block_n/2, (r+1)*block_n/2) of the B tile; the leader
  // issues tcgen05.mma.cta_group::2 (M = 256).  sm_tiles / total_tiles then count PAIR items.
  int pair;
};

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case GAP_ACT_LRELU:
      return v > 0.f ? v : 0.2f * v;
    case GAP_ACT_RELU:
      return fmaxf(v, 0.f);
    case GAP_ACT_TANH:
      return tanhf(v);
    case GAP_ACT_SIGMOID:
      return 1.f / (1.f + __expf(-v));
    default:
      return v;
  }
}

struct WorkCoord {
  int n_tile, sm, ph, pw, phase;
};
struct MTile {
  int tw, th, tn;
  bool exists;
};

__device__ __forceinline__ WorkCoord decode_work(const FpropParams& p, int t) {
  WorkCoord c;
  // N tile fastest, then the output-parity phase, then the M tile: the four phases of an M tile read the same input
  // window, so they run on neighbouring CTAs at the same time and share it in L2 (phase-major order re-read the
  // input from DRAM once per phase: 534 MB instead of 335 MB on the 128->64 dgrad, ncu dram__bytes_read).
  c.n_tile = t % p.n_tiles;
  t /= p.n_tiles;
  c.phase = t % p.n_phase;
  t /= p.n_phase;
  c.sm = t;
  c.ph = c.phase >> 1;
  c.pw = c.phase & 1;
  return c;
}
__device__ __forceinline__ MTile decode_mtile(const FpropParams& p, int mi) {
  MTile m;
  m.exists = mi < p.m_tiles_pp;
  m.tw = mi % p.tiles_w;
  mi /= p.tiles_w;
  m.th = mi % p.tiles_h;
  m.tn = mi / p.tiles_h;
  return m;
}

// Column sums of one 32-row x 16-column chunk on the warp MMA.  The chunk lives one row per lane as eight packed
// bf16 pairs (`a`, and `b` for the second factor; kSame: b == a).  The rows are staged in a 1 KiB smem tile
// (16-byte halves XOR-swizzled by bit 2 of the row so the 128-bit stores and the ldmatrix rows are conflict-free),
// read back transposed as MMA fragments, and reduced by   ones(16x32) * A   and   diag(B^T * A):
//   sum1[c] = sum_r a[r][c]          sum2[c] = sum_r a[r][c] * b[r][c]
// Products of bf16 pairs are exact in the fp32 accumulators.  Holder lanes l = 4m + (m >> 1), m = 0..7, receive
// out = {sum1[m], sum1[m+8], sum2[m], sum2[m+8]}; the other lanes receive unrelated values.
// Replaces two 31-shuffle transpose reductions (~140 instructions per chunk) by ~25.
template <bool kSame>
__device__ __forceinline__ void warp_colstats16(const uint32_t (&a)[8], const uint32_t (&b)[8], uint32_t stage,
                                                uint32_t lane, float (&out)[4]) {
  const uint32_t wr = stage + lane * 32u;
  const uint32_t wsw = ((lane >> 2) & 1u) << 4;
  const uint32_t mi = lane >> 3, rr = lane & 7u;
  const uint32_t row0 = (mi & 1u) * 8u + rr;  // + 16 for the second k block (bit 2 of the row is unchanged)
  const uint32_t rd = stage + row0 * 32u + ((((mi >> 1) & 1u) << 4) ^ (((row0 >> 2) & 1u) << 4));
  uint32_t qa[2][4], qb[2][4];
  __syncwarp();  // the previous chunk's fragment loads are done
  st_shared_v4(wr + wsw, a[0], a[1], a[2], a[3]);
  st_shared_v4(wr + (16u ^ wsw), a[4], a[5], a[6], a[7]);
  __syncwarp();
  ldmatrix_x4_trans(qa[0], rd);
  ldmatrix_x4_trans(qa[1], rd + 512u);
  if (!kSame) {
    __syncwarp();
    st_shared_v4(wr + wsw, b[0], b[1], b[2], b[3]);
    st_shared_v4(wr + (16u ^ wsw), b[4], b[5], b[6], b[7]);
    __syncwarp();
    ldmatrix_x4_trans(qb[0], rd);
    ldmatrix_x4_trans(qb[1], rd + 512u);
  }
  float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
  float q0[4] = {0.f, 0.f, 0.f, 0.f}, q1[4] = {0.f, 0.f, 0.f, 0.f};
  const uint32_t ones[4] = {0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u};
#pragma unroll
  for (int kb = 0; kb < 2; ++kb) {
    // fragments of the transposed loads: [0] rows 0-7 / cols 0-7, [1] rows 8-15 / cols 0-7, [2] rows 0-7 / cols 8-15,
    // [3] rows 8-15 / cols 8-15  ->  B fragments {[0],[1]} (cols 0-7), {[2],[3]} (cols 8-15); A = tile^T = {[0],[2],[1],[3]}
    const uint32_t(&fa)[4] = qa[kb];
    const uint32_t(&fb)[4] = kSame ? qa[kb] : qb[kb];
    const uint32_t at[4] = {fb[0], fb[2], fb[1], fb[3]};
    mma_bf16_16816(s0, ones, fa[0], fa[1]);
    mma_bf16_16816(s1, ones, fa[2], fa[3]);
    mma_bf16_16816(q0, at, fa[0], fa[1]);
    mma_bf16_16816(q1, at, fa[2], fa[3]);
  }
  const int sel = (lane >> 2) & 1;
  out[0] = sel ? s0[1] : s0[0];
  out[1] = sel ? s1[1] : s1[0];
  out[2] = sel ? q0[1] : q0[0];
  out[3] = sel ? q1[3] : q1[2];
}

// Cold path of the epilogue: partial column chunks, unaligned outputs, fp32 output, Tanh / Sigmoid.
// Kept out of line so the hot loop stays small (the inlined version was instruction-cache bound).
// The 16 values travel in registers (four float4 arguments): passing the array by reference made the compiler
// spill it to local memory on EVERY chunk of the hot path (4 STL.128 per chunk, as many L1 wavefronts as the
// backward epilogue's global loads -- ncu, profiles/r1_ncu_bwd_epilogue.md).
__device__ __noinline__ void epilogue_store_generic(const FpropParams& p, float4 v0, float4 v1, float4 v2, float4 v3,
                                                    long long pix, int col0) {
  const float f[16] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w};
  if (p.out_f32) {
    float* o = reinterpret_cast<float*>(p.out) + pix * p.out_ld + col0;
    for (int j = 0; j < 16; ++j)
      if (col0 + j < p.n_out) o[j] = apply_act(f[j], p.act) + (p.accum ? o[j] : 0.f);
    return;
  }
  for (int j = 0; j < 16; ++j) {
    if (col0 + j < p.n_out) {
      const float prev = p.accum ? __bfloat162float(p.out[pix * p.out_ld + col0 + j]) : 0.f;
      p.out[pix * p.out_ld + col0 + j] = __float2bfloat16(apply_act(f[j], p.act) + prev);
      if (p.out2 != nullptr) p.out2[pix * p.out2_ld + col0 + j] = __float2bfloat16(apply_act(f[j], p.act2));
    }
  }
}

template <int kEpi, bool kPair = false>
__global__ void __launch_bounds__(kFpropThreads, 1)
conv_fprop_kernel(const __grid_constant__ FpropParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  // pair mode: this CTA's half of the B rows; rank 0 (the leader) issues the MMAs for both CTAs
  const uint32_t cta_rank = kPair ? cluster_ctarank() : 0u;
  const int bn_cta = kPair ? (p.block_n >> 1) : p.block_n;
  const int tile0 = kPair ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = kPair ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int a_bytes = p.mt * p.a_tile_bytes;
  const int stage_bytes = a_bytes + p.b_per_stage * bn_cta * 128;
  const uint32_t bar_base = smem_base + p.num_stages * stage_bytes;
  // barrier slots (8 bytes each): full[0..7], empty[8..15], tfull[16..17], tempty[18..19]
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kMaxStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kMaxStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kMaxStages + 2 + a); };
  uint8_t* bar_gen = smem_gen + p.num_stages * stage_bytes;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bar_gen + 8 * 20);
  double* stats_sm = reinterpret_cast<double*>(bar_gen + kBarrierBytes);
  float* par_sm = reinterpret_cast<float*>(bar_gen + kBarrierBytes + kStatsBytes);  // [2][256] scale | shift
  const uint32_t colstage_base = bar_base + kBarrierBytes + kStatsBytes + kParamBytes;  // [kEpiWarps][1 KiB]

  // Warp index broadcast from lane 0: the role dispatch and the producer / MMA loops are then
  // warp-uniform for the compiler, so TMA / MMA operands stay in uniform registers (a per-lane
  // `if (lane == 0)` loop makes ptxas wrap every UTMALDG / UTCHMMA in a lane-serialising loop).
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const uint32_t lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmA[0]);
    if (p.src_chunks[1] > 0) tma_prefetch_desc(&p.tmA[1]);
    tma_prefetch_desc(&p.tmB);
    for (int s = 0; s < p.num_stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), kPair ? 2 * kEpiWarps : kEpiWarps);   // pair: both CTAs' epilogue warps release the leader
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (kPair) {
      tmem_alloc_pair(smem_u32(const_cast<uint32_t*>(tmem_slot)), kTmemCols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (kPair)
    cluster_sync();      // the peer's barriers are initialised before anything signals them
  else
    __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();   // the next kernel's CTAs may be scheduled as SMs drain; they block in their own pdl_wait()
  pdl_wait();      // everything above overlapped the previous kernel; its results are visible from here on

  const int BW = 1 << p.log_bw, BH = 1 << p.log_bh;
  const int BNI = kBlockM >> (p.log_bw + p.log_bh);
  const int n_taps = p.taps_h * p.taps_w;

  if (warp == 0 || warp == kProducer2Warp) {
    // ------------------------------------------------------------------ TMA producers
    // Two single-lane producers split the pipeline iterations even / odd: one lane needs ~280 cycles of fixed work per
    // iteration (mbarrier try_wait + expect_tx + address arithmetic, measured) plus ~50 per TMA, which is the bound for
    // small tiles (N <= 64, or the deep layers with 128 iterations of tiny MMAs).
    if (elect_one()) {
      const uint32_t my_par = warp == 0 ? 0u : 1u;
      uint32_t it = 0;
      int stage = 0;
      uint32_t phase = 0;
      // pair mode: every load reports its bytes to the LEADER's full barrier (the leader arms it for both CTAs); a
      // tile that does not exist is still fetched (its coordinates are out of range: zero fill, same byte count)
      auto ld_a = [&](uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
        if (kPair)
          tma_load_4d_pair(dst, tm, bar, c0, c1, c2, c3);
        else
          tma_load_4d(dst, tm, bar, c0, c1, c2, c3);
      };
      auto ld_b = [&](uint32_t dst, uint32_t bar, int c0, int c1, int c2) {
        if (kPair)
          tma_load_3d_pair(dst, &p.tmB, bar, c0, c1, c2);
        else
          tma_load_3d(dst, &p.tmB, bar, c0, c1, c2);
      };
      auto fbar = [&](int s) { return kPair ? mapa_cluster(full_bar(s), 0u) : full_bar(s); };
      for (int tile = tile0; tile < p.total_tiles; tile += tile_step) {
        const WorkCoord wc = decode_work(p, tile);
        const int sm_own = kPair ? (wc.sm * 2 + static_cast<int>(cta_rank)) : wc.sm;
        const MTile m0 = decode_mtile(p, sm_own * p.mt);
        const MTile m1 = decode_mtile(p, sm_own * p.mt + 1);
        const bool has1 = p.mt > 1 && (m1.exists || kPair);
        const int x0 = m0.tw * BW * p.in_stride + p.in_off_w[wc.pw];
        const int y0 = m0.th * BH * p.in_stride + p.in_off_h[wc.ph];
        const int n0 = m0.tn * BNI;
        const int x1 = m1.tw * BW * p.in_stride + p.in_off_w[wc.pw];
        const int y1 = m1.th * BH * p.in_stride + p.in_off_h[wc.ph];
        const int n1 = m1.tn * BNI;
        // bytes one CTA receives per stage; the leader of a pair arms its barrier for both CTAs
        const uint32_t tx_bytes =
            static_cast<uint32_t>(bn_cta * 128 + (has1 ? 2 : 1) * kATileBytes) * (kPair ? 2u : 1u);
        const int b_row = wc.n_tile * p.block_n + static_cast<int>(cta_rank) * bn_cta;
        const bool arm = !kPair || cta_rank == 0;
        if (p.halo) {
          const uint32_t txh =
              static_cast<uint32_t>(p.halo_taps * bn_cta * 128 + (has1 ? 2 : 1) * p.a_load_bytes) * (kPair ? 2u : 1u);
          for (int t_w = 0; t_w < p.taps_w; ++t_w) {
            for (int g = 0; g < p.halo_groups; ++g) {
              int cc = 0;
              for (int s = 0; s < 2; ++s) {
                for (int c = 0; c < p.src_chunks[s]; ++c, ++cc) {
                  if ((it++ & 1u) == my_par) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    if (arm) mbar_expect_tx(full_bar(stage), txh);
                    const uint32_t fb = fbar(stage);
                    const uint32_t a_dst = smem_base + stage * stage_bytes;
                    ld_a(a_dst, &p.tmA[s], fb, c * kBlockK, x0 + t_w, y0 + g, n0);
                    if (has1) ld_a(a_dst + p.a_tile_bytes, &p.tmA[s], fb, c * kBlockK, x1 + t_w, y1 + g, n1);
                    for (int i = 0; i < p.halo_taps; ++i) {
                      const int t_h = g + p.halo_groups * i;
                      ld_b(a_dst + a_bytes + i * bn_cta * 128, fb, ((t_h * p.taps_w + t_w) * p.chunks_tot + cc) * kBlockK,
                           b_row, wc.phase);
                    }
                  }
                  if (++stage == p.num_stages) {
                    stage = 0;
                    phase ^= 1u;
                  }
                }
              }
            }
          }
          continue;
        }
        int kcol = 0;
        for (int t_h = 0; t_h < p.taps_h; ++t_h) {
          for (int t_w = 0; t_w < p.taps_w; ++t_w) {
            for (int s = 0; s < 2; ++s) {
              for (int c = 0; c < p.src_chunks[s]; ++c) {
                if ((it++ & 1u) == my_par) {
                  mbar_wait(empty_bar(stage), phase ^ 1u);
                  if (arm) mbar_expect_tx(full_bar(stage), tx_bytes);
                  const uint32_t fb = fbar(stage);
                  const uint32_t a_dst = smem_base + stage * stage_bytes;
                  ld_a(a_dst, &p.tmA[s], fb, c * kBlockK, x0 + t_w, y0 + t_h, n0);
                  if (has1) ld_a(a_dst + kATileBytes, &p.tmA[s], fb, c * kBlockK, x1 + t_w, y1 + t_h, n1);
                  ld_b(a_dst + a_bytes, fb, kcol, b_row, wc.phase);
                }
                kcol += kBlockK;
                if (++stage == p.num_stages) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (pair mode: the leader CTA only)
    auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t accum) {
      if (kPair)
        umma_bf16_pair(d, ad, bd, p.idesc, accum);
      else
        umma_bf16(d, ad, bd, p.idesc, accum);
    };
    auto commit = [&](uint32_t bar) {      // pair mode: the arrival lands on the same barrier of BOTH CTAs
      if (kPair)
        umma_commit_pair(bar, 0x3);
      else
        umma_commit(bar);
    };
    if ((!kPair || cta_rank == 0) && elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = tile0; tile < p.total_tiles; tile += tile_step) {
        const WorkCoord wc = decode_work(p, tile);
        const int mt_eff = kPair ? p.mt : min(p.mt, p.m_tiles_pp - wc.sm * p.mt);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccStride;
        for (int k_iter = 0; k_iter < p.k_iters; ++k_iter) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t a_addr = smem_base + stage * stage_bytes;
          const uint32_t b_addr = a_addr + a_bytes;
          if (p.halo) {
            const uint32_t row_shift = static_cast<uint32_t>(128 << p.log_bw);   // one input row of the tile = BW pixels
            for (int j = 0; j < mt_eff; ++j) {
              for (int i = 0; i < p.halo_taps; ++i) {
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                  const uint64_t adesc = make_sw128_desc(a_addr + j * p.a_tile_bytes + i * row_shift + k * 32, 16, 1024);
                  const uint64_t bdesc = make_sw128_desc(b_addr + i * bn_cta * 128 + k * 32, 16, 1024);
                  mma(d_tmem + j * p.block_n, adesc, bdesc, (k_iter | i | k) != 0 ? 1u : 0u);
                }
              }
            }
          } else {
            for (int j = 0; j < mt_eff; ++j) {
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k) {
                const uint64_t adesc = make_sw128_desc(a_addr + j * kATileBytes + k * 32, 16, 1024);
                const uint64_t bdesc = make_sw128_desc(b_addr + k * 32, 16, 1024);
                mma(d_tmem + j * p.block_n, adesc, bdesc, (k_iter | k) != 0 ? 1u : 0u);
              }
            }
          }
          commit(empty_bar(stage));
          if (++stage == p.num_stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        commit(tfull_bar(acc));
        if (++acc == p.acc_stages) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..9)
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;  // the two warps of a quarter take the even / odd 16-column chunks
    const int row = q * 32 + lane;
    const int e_tid = threadIdx.x - 64;  // 0..255
    int acc = 0;
    uint32_t acc_phase = 0;
    int cur_ntile = -1;
    double* my_stats = stats_sm + q * 512;  // [256 sum][256 sumsq]
    const bool do_stats = p.stats != nullptr && !(p.skip & 4);
    const uint32_t colstage = colstage_base + static_cast<uint32_t>(warp - 2) * 1024u;
    const bool stat_holder = (lane >> 3) == (lane & 3u);  // lanes 4m + (m >> 1): columns m and m + 8 of a chunk
    const int stat_col = static_cast<int>(lane >> 2);

    auto flush_stats = [&](int n_tile) {
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int c = e_tid; c < 2 * p.block_n; c += 32 * kEpiWarps) {
        const int which = c / p.block_n, col = c - which * p.block_n;
        const int gcol = n_tile * p.block_n + col;
        const int idx = which * 256 + col;
        double tot = stats_sm[idx] + stats_sm[512 + idx] + stats_sm[1024 + idx] + stats_sm[1536 + idx];
        if (kEpi == 1) {
          const int n_stats = p.n_out - p.bwd_c0;
          if (gcol >= p.bwd_c0 && gcol < p.n_out) atomicAdd(p.stats + which * n_stats + (gcol - p.bwd_c0), tot);
        } else if (gcol < p.n_out) {
          atomicAdd(p.stats + which * p.n_out + gcol, tot);
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
    };

    for (int tile = tile0; tile < p.total_tiles; tile += tile_step) {
      const WorkCoord wc = decode_work(p, tile);
      const int sm_own = kPair ? (wc.sm * 2 + static_cast<int>(cta_rank)) : wc.sm;
      if ((do_stats || kEpi == 1) && wc.n_tile != cur_ntile) {
        if (do_stats && cur_ntile >= 0) flush_stats(cur_ntile);
        if (do_stats) {
          if (half == 0)
            for (int c = lane; c < 512; c += 32) my_stats[c] = 0.0;
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        if (kEpi == 1) {
          // stage this N tile's BatchNorm scale / shift (identity when the layer has no BatchNorm)
          if (!do_stats) asm volatile("bar.sync 1, 256;" ::: "memory");  // previous tile's readers are done
          for (int c = e_tid; c < p.block_n; c += 32 * kEpiWarps) {
            const int gcol = wc.n_tile * p.block_n + c;
            const bool on = p.bwd_scale != nullptr && gcol >= p.bwd_c0 && gcol < p.n_out;
            par_sm[c] = on ? __ldg(p.bwd_scale + gcol - p.bwd_c0) : 1.f;
            par_sm[256 + c] = on ? __ldg(p.bwd_shift + gcol - p.bwd_c0) : 0.f;
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        __syncwarp();
        cur_ntile = wc.n_tile;
      }
      // (Tried: prefetch.global.L2 of the next work item's y / g2 rows here.  5 % SLOWER: the loads wait on the L1
      // data pipe, which the tensor-core operand reads and TMA writes keep ~70 % busy, not on DRAM.)
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const int n_chunks = p.block_n >> 4;
      for (int j = 0; j < p.mt; ++j) {
        const MTile mtile = decode_mtile(p, sm_own * p.mt + j);
        const int wi = row & (BW - 1);
        const int hi = (row >> p.log_bw) & (BH - 1);
        const int ni = row >> (p.log_bw + p.log_bh);
        const int gx = mtile.tw * BW + wi, gy = mtile.th * BH + hi, n = mtile.tn * BNI + ni;
        const bool valid = mtile.exists && (gx < p.gw) && (gy < p.gh) && (n < p.n_img);
        const long long pix =
            (static_cast<long long>(n) * p.OH + (gy * p.out_stride + wc.ph)) * p.OW + (gx * p.out_stride + wc.pw);
        const uint32_t t_row =
            tmem_base + acc * kAccStride + j * p.block_n + (static_cast<uint32_t>(q * 32) << 16);
        if (!mtile.exists) continue;
        const bool fast = valid && p.fast_store;
        for (int cg = half; cg < n_chunks; cg += 8) {
          // backward-fused epilogue: issue the y / g2 loads of up to four chunks before touching TMEM, so their
          // latency overlaps (the epilogue is latency-bound otherwise: only four warps per CTA)
          uint4 yq[4][2], gq[4][2];
          if (kEpi == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              yq[i][0] = yq[i][1] = gq[i][0] = gq[i][1] = make_uint4(0, 0, 0, 0);
              const int colp = wc.n_tile * p.block_n + (cg + 2 * i) * 16;
              if (valid && cg + 2 * i < n_chunks && colp >= p.bwd_c0 && colp < p.n_out && !(p.skip & 2)) {
                const __nv_bfloat16* yp = p.bwd_y + pix * p.bwd_y_ld + (colp - p.bwd_c0);
                if (p.bwd_ld32) {
                  ld_global_nc_32B(yp, yq[i][0], yq[i][1]);
                } else {
                  yq[i][0] = __ldg(reinterpret_cast<const uint4*>(yp));
                  yq[i][1] = __ldg(reinterpret_cast<const uint4*>(yp) + 1);
                }
                if (p.bwd_g2 != nullptr) {
                  const __nv_bfloat16* gp = p.bwd_g2 + pix * p.bwd_g2_ld + (colp - p.bwd_c0);
                  if (p.bwd_ld32) {
                    ld_global_nc_32B(gp, gq[i][0], gq[i][1]);
                  } else {
                    gq[i][0] = __ldg(reinterpret_cast<const uint4*>(gp));
                    gq[i][1] = __ldg(reinterpret_cast<const uint4*>(gp) + 1);
                  }
                }
              }
            }
          }
          if (kEpi == 2) {
            // accumulate mode: the values already in `out`, fetched the same way (coherent loads: this thread
            // overwrites them below)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              yq[i][0] = yq[i][1] = make_uint4(0, 0, 0, 0);
              const int colp = wc.n_tile * p.block_n + (cg + 2 * i) * 16;
              if (fast && cg + 2 * i < n_chunks && colp + 16 <= p.n_out)
                ld_global_32B(p.out + pix * p.out_ld + colp, yq[i][0], yq[i][1]);
            }
          }
#pragma unroll
          for (int ci = 0; ci < 4; ++ci) {
          const int c = cg + 2 * ci;
          if (c >= n_chunks) break;
          uint32_t raw[16];
          tmem_ld16(t_row + c * 16, raw);
          tmem_ld_wait();
          const int col0 = wc.n_tile * p.block_n + c * 16;
          float f[16];
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) f[jj] = __uint_as_float(raw[jj]);
          if (kEpi == 1 && col0 >= p.bwd_c0) {
            // d = mask(y) ? g (+ g2) : slope * g  with mask = (y*scale + shift > 0); sums of d and d*y
            const uint32_t* yw = reinterpret_cast<const uint32_t*>(yq[ci]);
            const uint32_t* gw = reinterpret_cast<const uint32_t*>(gq[ci]);
            const float4* scp = reinterpret_cast<const float4*>(par_sm + c * 16);
            const float4* shp = reinterpret_cast<const float4*>(par_sm + 256 + c * 16);
            float yv[16];
#pragma unroll
            for (int v4 = 0; v4 < 4; ++v4) {
              float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
              if (p.bwd_scale != nullptr) {   // no BatchNorm below: the mask is just y > 0, skip the smem reads
                sc = scp[v4];
                sh = shp[v4];
              }
              const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int jj = v4 * 4 + e;
                const uint32_t ywd = yw[jj >> 1], gwd = gw[jj >> 1];
                const float y = (jj & 1) ? bf16_hi(ywd) : bf16_lo(ywd);
                const float g2 = (jj & 1) ? bf16_hi(gwd) : bf16_lo(gwd);
                yv[jj] = y;
                const float yh = fmaf(y, scv[e], shv[e]);
                f[jj] = yh > 0.f ? f[jj] + g2 : p.bwd_slope * f[jj];
              }
            }
            uint32_t pk[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) pk[jj] = valid ? pack_bf16x2(f[2 * jj], f[2 * jj + 1]) : 0u;
            if (do_stats) {
              // sums of d and d*y over the 32 rows, from the bf16 values that are stored / were loaded
              uint32_t yk[8];
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) yk[jj] = yw[jj];
              float cs[4];
              warp_colstats16<false>(pk, yk, colstage, lane, cs);
              if (stat_holder) {
                my_stats[c * 16 + stat_col] += static_cast<double>(cs[0]);
                my_stats[c * 16 + stat_col + 8] += static_cast<double>(cs[1]);
                my_stats[256 + c * 16 + stat_col] += static_cast<double>(cs[2]);
                my_stats[256 + c * 16 + stat_col + 8] += static_cast<double>(cs[3]);
              }
            }
            // n_tiles * block_n can exceed n_out (272 = 2 x 144, 640 = 3 x 224): the chunks past the last channel are
            // whole (n_out - c0 and c0 are multiples of 16) and are not stored
            if (valid && col0 < p.n_out && !(p.skip & 1)) st_global_32B(p.out + pix * p.out_ld + col0, pk, true);
            continue;
          }
          if (p.scale != nullptr) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) f[jj] *= __ldg(p.scale + min(col0 + jj, p.n_out - 1));
          }
          if (p.bias != nullptr) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) f[jj] += __ldg(p.bias + min(col0 + jj, p.n_out - 1));
          }
          if (do_stats && kEpi != 1) {
            // BatchNorm batch statistics (sum, sum of squares) of the bf16-rounded pre-activation values
            uint32_t pr[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) pr[jj] = valid ? pack_bf16x2(f[2 * jj], f[2 * jj + 1]) : 0u;
            float cs[4];
            warp_colstats16<true>(pr, pr, colstage, lane, cs);
            if (stat_holder) {
              my_stats[c * 16 + stat_col] += static_cast<double>(cs[0]);
              my_stats[c * 16 + stat_col + 8] += static_cast<double>(cs[1]);
              my_stats[256 + c * 16 + stat_col] += static_cast<double>(cs[2]);
              my_stats[256 + c * 16 + stat_col + 8] += static_cast<double>(cs[3]);
            }
          }
          if (fast && col0 + 16 <= p.n_out && !(p.skip & 1)) {
            // common case: slope-type activation (identity / LeakyReLU / ReLU), 256-bit stores
            uint32_t pk[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              const float a0 = f[2 * jj], a1 = f[2 * jj + 1];
              float v0 = a0 * (a0 > 0.f ? 1.f : p.slope1), v1 = a1 * (a1 > 0.f ? 1.f : p.slope1);
              if (kEpi == 2) {
                const uint32_t prev = reinterpret_cast<const uint32_t*>(yq[ci])[jj];
                v0 += bf16_lo(prev);
                v1 += bf16_hi(prev);
              }
              pk[jj] = pack_bf16x2(v0, v1);
            }
            st_global_32B(p.out + pix * p.out_ld + col0, pk, true);
            if (p.out2 != nullptr) {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
                const float a0 = f[2 * jj], a1 = f[2 * jj + 1];
                pk[jj] = pack_bf16x2(a0 * (a0 > 0.f ? 1.f : p.slope2), a1 * (a1 > 0.f ? 1.f : p.slope2));
              }
              st_global_32B(p.out2 + pix * p.out2_ld + col0, pk, true);
            }
          } else if (valid && col0 < p.n_out) {
            epilogue_store_generic(p, make_float4(f[0], f[1], f[2], f[3]), make_float4(f[4], f[5], f[6], f[7]),
                                   make_float4(f[8], f[9], f[10], f[11]), make_float4(f[12], f[13], f[14], f[15]), pix,
                                   col0);
          }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kPair)
          mbar_arrive_cluster(mapa_cluster(tempty_bar(acc), 0u));     // the leader's MMA lane waits for both CTAs
        else
          mbar_arrive(tempty_bar(acc));
      }
      if (++acc == p.acc_stages) {
        acc = 0;
        acc_phase ^= 1u;
      }
    }
    if (do_stats && cur_ntile >= 0) flush_stats(cur_ntile);
  }

  tc_fence_before();
  if (kPair)
    cluster_sync();      // neither CTA frees its TMEM / exits while the peer's MMAs or remote arrivals may still touch it
  else
    __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (kPair)
      tmem_dealloc_pair(tmem_base, kTmemCols);
    else
      tmem_dealloc(tmem_base, kTmemCols);
  }
}

static int ilog2_ceil(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

}  // namespace gap

using namespace gap;

extern "C" int gap_conv_gemm(const gap_conv_gemm_args* a, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  GAP_CHECK_ARG(a != nullptr, "gap_conv_gemm: null args");
  GAP_CHECK_ARG(a->src[0] && a->wpk && a->out, "gap_conv_gemm: null src/wpk/out pointer");
  GAP_CHECK_ARG(a->src_c[0] > 0 && a->src_c[0] % 64 == 0 && a->src_c[1] >= 0 &&
                    a->src_c[1] % 64 == 0,
                "gap_conv_gemm: source channels (%d, %d) must be multiples of 64", a->src_c[0],
                a->src_c[1]);
  GAP_CHECK_ARG(a->src_c[1] == 0 || a->src[1] != nullptr, "gap_conv_gemm: src[1] is null");
  GAP_CHECK_ARG(a->n > 0 && a->ih > 0 && a->iw > 0 && a->gh > 0 && a->gw > 0,
                "gap_conv_gemm: empty shape n=%d ih=%d iw=%d gh=%d gw=%d", a->n, a->ih, a->iw,
                a->gh, a->gw);
  GAP_CHECK_ARG(a->n_phase == 1 || a->n_phase == 4, "gap_conv_gemm: n_phase must be 1 or 4");
  GAP_CHECK_ARG(a->taps_h >= 1 && a->taps_w >= 1 && a->taps_h <= 7 && a->taps_w <= 7,
                "gap_conv_gemm: taps out of range");
  GAP_CHECK_ARG(a->in_stride >= 1 && a->in_stride <= 2 && a->out_stride >= 1,
                "gap_conv_gemm: strides out of range");
  GAP_CHECK_ARG(a->n_out >= 1 && a->w_rows >= a->n_out, "gap_conv_gemm: n_out/w_rows invalid");
  GAP_CHECK_ARG(a->act >= 0 && a->act <= 4 && a->act2 >= 0 && a->act2 <= 4,
                "gap_conv_gemm: unknown activation");
  for (int s = 0; s < 2; ++s) {
    if (a->src_c[s] == 0) continue;
    if (a->src_ld[s] < a->src_c[s] || a->src_ld[s] % 8 != 0) {
      set_error("gap_conv_gemm: src_ld[%d]=%lld must be >= channels and a multiple of 8", s,
                (long long)a->src_ld[s]);
      return GAP_ERR_ALIGNMENT;
    }
  }
  const bool vec_ok =
      a->out_ld % 8 == 0 && (reinterpret_cast<uintptr_t>(a->out) & 15) == 0 &&
      (!a->out2 || (a->out2_ld % 8 == 0 && (reinterpret_cast<uintptr_t>(a->out2) & 15) == 0));

  FpropParams p;
  memset(&p, 0, sizeof(p));
  // ---- M tile shape
  int log_bw = std::min(7, ilog2_ceil(a->gw));
  int log_bh = std::min(7 - log_bw, ilog2_ceil(a->gh));
  // Halo mode (see FpropParams): needs a tile inside one image whose width is a multiple of 8 pixels and at least
  // two taps that differ by whole input rows; the N tile must be small enough for halo_taps B tiles per stage
  // (checked below, after block_n is known).
  const int halo_taps = a->taps_h / a->in_stride;
  bool halo = debug_get("fprop_halo", 1) != 0 && halo_taps >= 2 && a->taps_h % a->in_stride == 0;
  if (halo) {
    if (a->gw >= 16 && a->gh >= 8) {
      log_bw = 4;
      log_bh = 3;
    } else if (a->gw >= 8 && a->gh >= 16) {
      log_bw = 3;
      log_bh = 4;
    } else {
      halo = false;
    }
  }
  const int n_pad_h = (a->n_out + 15) / 16 * 16;
  if (halo && std::min(n_pad_h, 256) * halo_taps > 256) {
    halo = false;     // would need more than 32 KiB of B tiles per stage: these layers are B-traffic bound anyway
    log_bw = std::min(7, ilog2_ceil(a->gw));
    log_bh = std::min(7 - log_bw, ilog2_ceil(a->gh));
  }
  const int BW = 1 << log_bw, BH = 1 << log_bh, BNI = kBlockM / (BW * BH);
  p.log_bw = log_bw;
  p.log_bh = log_bh;
  p.tiles_w = (a->gw + BW - 1) / BW;
  p.tiles_h = (a->gh + BH - 1) / BH;
  p.tiles_n = (a->n + BNI - 1) / BNI;
  const int m_tiles_pp = p.tiles_w * p.tiles_h * p.tiles_n;
  const int m_tiles = m_tiles_pp * a->n_phase;
  // ---- N tile
  const int n_pad = (a->n_out + 15) / 16 * 16;
  int n_tiles = (n_pad + 255) / 256;
  int block_n = ((n_pad + n_tiles - 1) / n_tiles + 15) / 16 * 16;
  const int sms = sm_count();
  const int force_bn = debug_get("fprop_block_n", 0);
  int model_mt = 0;
  if (force_bn > 0) {
    block_n = force_bn;
    n_tiles = (n_pad + block_n - 1) / block_n;
  } else if (!halo && m_tiles * n_tiles < 2 * sms) {
    // Under-filled launch (the 8x8 .. 1x1 bottleneck layers): every CTA runs one or two latency-bound K loops, so
    // pick the N tile and the M tiles per item by a per-iteration cost model fitted to tools/sweep_deep.py:
    // cycles per pipeline iteration ~ max(130 + 280 per A tile + 80 per 64 B rows, MMA time 2*mt*bn + 100), times
    // the number of waves.  (The old rule halved block_n until every SM had an item: up to 2x slower.)
    const int wide = block_n;
    long long best = -1;
    for (int bn_c : {wide, 128, 64}) {
      if (bn_c > wide || (bn_c != wide && wide % bn_c != 0)) continue;
      for (int mt_c = 1; mt_c <= 2; ++mt_c) {
        if (mt_c == 2 && m_tiles_pp < 2) continue;
        const long long items =
            static_cast<long long>((m_tiles_pp + mt_c - 1) / mt_c) * a->n_phase * ((n_pad + bn_c - 1) / bn_c);
        const long long waves = (items + sms - 1) / sms;
        const long long it_cost = std::max(130 + 280 * mt_c + 80 * bn_c / 64, 2 * mt_c * bn_c + 100);
        const long long cost = waves * it_cost;
        if (best < 0 || cost < best) {
          best = cost;
          block_n = bn_c;
          model_mt = mt_c;
        }
      }
    }
    n_tiles = (n_pad + block_n - 1) / block_n;
  }
  const int k_iters_full = a->taps_h * a->taps_w * ((a->src_c[0] + a->src_c[1]) / 64);
  // Two M tiles per work item share each B tile (halves the weight traffic from L2) when there is
  // still at least ~2 waves of work items left.
  int mt = (m_tiles_pp >= 2 && (m_tiles / 2) * n_tiles >= 2 * sms) ? 2 : 1;
  // With a 256-wide N tile two M tiles fill all 512 TMEM columns, so the epilogue cannot overlap the next item's
  // main loop: that only pays for long K loops (tools/sweep_mt.py: mt = 1 is 5-17 % faster below 128 iterations).
  if (mt == 2 && 2 * block_n > kAccStride && k_iters_full < 128) mt = 1;
  if (model_mt > 0) mt = model_mt;
  const int force_mt = debug_get("fprop_mt", 0);
  if (force_mt > 0) mt = std::min(force_mt, 2);
  // CTA pairs (cta_group::2, see FpropParams::pair): per SM half of every B tile is written by TMA and read by the tensor
  // core.  MEASURED per layer (profiles/r2_pair_mode_per_layer.txt, serialised launches of the batch-64 step): the
  // 256-wide N tiles with long K loops gain 1.5-6 % (512->256 s1: 1323 -> 1353 TFLOP/s, 256->1024: 1189 -> 1258), the
  // N <= 128 and four-phase layers LOSE 3-12 % (the two CTAs run in lock step and every release crosses the cluster),
  // so pairs are used only for single-phase launches with a 256-wide N tile, >= 64 K iterations and enough work items
  // for every cluster.  fprop_pair = 2 forces pairs wherever they are legal (tests, A/B runs), 0 disables them.
  const int pair_knob = debug_get("fprop_pair", 1);
  bool pair = pair_knob != 0 && sms % 2 == 0 && block_n % 16 == 0 && block_n >= 32 && !a->accumulate;
  if (pair && pair_knob != 2 && !(block_n == 256 && a->n_phase == 1 && k_iters_full >= 64)) pair = false;
  if (pair) {
    const long long pair_items = static_cast<long long>((m_tiles_pp + 2 * mt - 1) / (2 * mt)) * a->n_phase * n_tiles;
    if (pair_items < sms / 2) pair = false;
  }
  p.pair = pair ? 1 : 0;
  p.mt = mt;
  p.m_tiles_pp = m_tiles_pp;
  p.sm_tiles = pair ? (m_tiles_pp + 2 * mt - 1) / (2 * mt) : (m_tiles_pp + mt - 1) / mt;
  p.acc_stages = (mt * block_n <= kAccStride) ? 2 : 1;
  p.block_n = block_n;
  p.n_tiles = n_tiles;
  p.total_tiles = p.sm_tiles * a->n_phase * n_tiles;
  const int ctot = a->src_c[0] + a->src_c[1];
  p.src_chunks[0] = a->src_c[0] / 64;
  p.src_chunks[1] = a->src_c[1] / 64;
  p.k_iters = a->taps_h * a->taps_w * (ctot / 64);
  p.chunks_tot = ctot / 64;
  const int halo_rows = BH + halo_taps - 1;
  p.halo = halo ? 1 : 0;
  p.halo_taps = halo ? halo_taps : 1;
  p.halo_groups = halo ? a->in_stride : 1;
  p.a_load_bytes = halo ? halo_rows * BW * 128 : kATileBytes;
  p.a_tile_bytes = halo ? (p.a_load_bytes + 1023) / 1024 * 1024 : kATileBytes;
  p.b_per_stage = halo ? halo_taps : 1;
  if (halo) p.k_iters = a->taps_w * a->in_stride * (ctot / 64);
  p.n_img = a->n;
  p.gh = a->gh;
  p.gw = a->gw;
  p.n_phase = a->n_phase;
  p.taps_h = a->taps_h;
  p.taps_w = a->taps_w;
  p.in_stride = a->in_stride;
  for (int i = 0; i < 2; ++i) {
    p.in_off_h[i] = a->in_off_h[i];
    p.in_off_w[i] = a->in_off_w[i];
  }
  p.out_stride = a->out_stride;
  p.n_out = a->n_out;
  p.OH = a->oh;
  p.OW = a->ow;
  p.out = static_cast<__nv_bfloat16*>(a->out);
  p.out_ld = a->out_ld;
  p.act = a->act;
  p.out2 = static_cast<__nv_bfloat16*>(a->out2);
  p.out2_ld = a->out2_ld;
  p.act2 = a->act2;
  p.bias = a->bias;
  p.scale = a->scale;
  p.stats = a->stats;
  p.idesc = make_idesc_bf16(pair ? 2 * kBlockM : kBlockM, block_n, 0, 0);
  const bool vec32 =
      vec_ok && a->out_ld % 16 == 0 && (reinterpret_cast<uintptr_t>(a->out) & 31) == 0 &&
      (!a->out2 || (a->out2_ld % 16 == 0 && (reinterpret_cast<uintptr_t>(a->out2) & 31) == 0));
  p.vec_ok = vec32 ? 2 : (vec_ok ? 1 : 0);
  p.out_f32 = a->out_f32;
  auto slope_of = [](int act) { return act == GAP_ACT_NONE ? 1.f : (act == GAP_ACT_LRELU ? 0.2f : 0.f); };
  p.slope1 = slope_of(a->act);
  p.slope2 = slope_of(a->act2);
  p.fast_store = (vec32 && !a->out_f32 && a->act <= GAP_ACT_RELU && a->act2 <= GAP_ACT_RELU) ? 1 : 0;
  GAP_CHECK_ARG(!(a->out_f32 && a->out2), "gap_conv_gemm: out2 is not supported with fp32 output");
  const bool bwd = a->bwd_y != nullptr;
  if (bwd) {
    const bool ok = vec32 && !a->out_f32 && !a->out2 && a->act == GAP_ACT_NONE && !a->bias && !a->scale && a->bwd_c0 >= 0 &&
                    a->bwd_c0 % 16 == 0 && a->bwd_c0 < a->n_out && (a->n_out - a->bwd_c0) % 16 == 0 &&
                    a->bwd_y_ld % 8 == 0 && (reinterpret_cast<uintptr_t>(a->bwd_y) & 15) == 0 &&
                    (!a->bwd_g2 || (a->bwd_g2_ld % 8 == 0 && (reinterpret_cast<uintptr_t>(a->bwd_g2) & 15) == 0)) &&
                    ((a->bwd_scale == nullptr) == (a->bwd_shift == nullptr));
    if (!ok) {
      set_error("gap_conv_gemm: the backward-fused epilogue needs a 32-byte aligned bf16 output without bias / "
                "activation / out2, 16-aligned channel ranges and 16-byte aligned y / g2 rows");
      return GAP_ERR_UNSUPPORTED;
    }
  }
  p.bwd_y = static_cast<const __nv_bfloat16*>(a->bwd_y);
  p.bwd_y_ld = a->bwd_y_ld;
  p.bwd_scale = a->bwd_scale;
  p.bwd_shift = a->bwd_shift;
  p.bwd_g2 = static_cast<const __nv_bfloat16*>(a->bwd_g2);
  p.bwd_g2_ld = a->bwd_g2_ld;
  p.bwd_slope = a->bwd_slope;
  p.bwd_c0 = a->bwd_c0;
  // 256-bit y / g2 loads when every chunk start is 32-byte aligned
  p.bwd_ld32 = (bwd && a->bwd_y_ld % 16 == 0 && (reinterpret_cast<uintptr_t>(a->bwd_y) & 31) == 0 &&
                (!a->bwd_g2 || (a->bwd_g2_ld % 16 == 0 && (reinterpret_cast<uintptr_t>(a->bwd_g2) & 31) == 0)) &&
                debug_get("fprop_ld32", 1) != 0)
                   ? 1
                   : 0;
  p.skip = debug_get("fprop_skip", 0);
  p.accum = a->accumulate ? 1 : 0;
  GAP_CHECK_ARG(!(a->accumulate && (bwd || a->out2 || a->stats)),
                "gap_conv_gemm: accumulate excludes the backward-fused epilogue, out2 and stats");

  const int stage_bytes = mt * p.a_tile_bytes + p.b_per_stage * (pair ? block_n / 2 : block_n) * 128;
  int stages = (kSmemBudget - 1024 - kBarrierBytes - kStatsBytes - kParamBytes - kColStageBytes) / stage_bytes;
  stages = std::min(stages, kMaxStages);
  const int force_st = debug_get("fprop_stages", 0);
  if (force_st > 0) stages = std::min(force_st, stages);
  p.num_stages = stages;
  const size_t smem_bytes = 1024 + static_cast<size_t>(stages) * stage_bytes + kBarrierBytes + kStatsBytes + kParamBytes + kColStageBytes;

  // ---- tensor maps
  const uint32_t bx_w = static_cast<uint32_t>(BW * a->in_stride);
  const uint32_t bx_h = static_cast<uint32_t>((halo ? halo_rows : BH) * a->in_stride);
  if (bx_w > 256 || bx_h > 256) {
    set_error("gap_conv_gemm: TMA box %ux%u exceeds 256", bx_w, bx_h);
    return GAP_ERR_UNSUPPORTED;
  }
  for (int s = 0; s < 2; ++s) {
    if (a->src_c[s] == 0) continue;
    const uint64_t ld_b = static_cast<uint64_t>(a->src_ld[s]) * 2;
    uint64_t dims[4] = {static_cast<uint64_t>(a->src_c[s]), static_cast<uint64_t>(a->iw),
                        static_cast<uint64_t>(a->ih), static_cast<uint64_t>(a->n)};
    uint64_t strides[3] = {ld_b, ld_b * a->iw, ld_b * a->iw * a->ih};
    uint32_t box[4] = {64, bx_w, bx_h, static_cast<uint32_t>(BNI)};
    uint32_t es[4] = {1, static_cast<uint32_t>(a->in_stride), static_cast<uint32_t>(a->in_stride), 1};
    int rc = encode_tmap_bf16(&p.tmA[s], a->src[s], 4, dims, strides, box, es, true);
    if (rc) return rc;
  }
  {
    const uint64_t ktot = static_cast<uint64_t>(a->taps_h) * a->taps_w * ctot;
    uint64_t dims[3] = {ktot, static_cast<uint64_t>(a->w_rows), static_cast<uint64_t>(a->n_phase)};
    uint64_t strides[2] = {ktot * 2, ktot * 2 * a->w_rows};
    uint32_t box[3] = {64, static_cast<uint32_t>(pair ? block_n / 2 : block_n), 1};
    int rc = encode_tmap_bf16(&p.tmB, a->wpk, 3, dims, strides, box, nullptr, true);
    if (rc) return rc;
  }

  static bool attr_set = false;
  if (!attr_set) {
    GAP_CUDA(cudaFuncSetAttribute(conv_fprop_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
    GAP_CUDA(cudaFuncSetAttribute(conv_fprop_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
    GAP_CUDA(cudaFuncSetAttribute(conv_fprop_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
    GAP_CUDA(cudaFuncSetAttribute(conv_fprop_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
    GAP_CUDA(cudaFuncSetAttribute(conv_fprop_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
    attr_set = true;
  }
  // Persistent grid: with W = ceil(items / slots) passes over the work list, ceil(items / W) CTAs finish at the same
  // time as `slots` would (the 3.46-wave launches of the 512-tile layers: 128 CTAs x 4 items instead of 148 CTAs of which
  // 80 idle through the last pass) and leave the other SMs to the kernels of the concurrent streams (weight gradients,
  // the generator forward next to the discriminator).  fprop_balance = 0: one CTA per SM as before.  Measured on the
  // whole iteration (tools/ab_knob.py, ABBA): 7.888 -> 7.842 ms.  (Also tried: walking the work list from the last M
  // tile down so that a conv reads first what the BatchNorm pass before it wrote last, i.e. what is still in L2:
  // 7.879 vs 7.875 ms, no effect -- the GEMMs are not DRAM-bound -- not kept.)
  auto balanced = [&](int items, int slots) {
    if (items <= slots || debug_get("fprop_balance", 1) == 0) return std::min(items, slots);
    const int passes = (items + slots - 1) / slots;
    return (items + passes - 1) / passes;
  };
  if (pair) {
    const int grid2 = 2 * balanced(p.total_tiles, sms / 2);
    if (bwd)
      GAP_CUDA(launch_pair(conv_fprop_kernel<1, true>, dim3(grid2), dim3(kFpropThreads), smem_bytes, stream, p));
    else
      GAP_CUDA(launch_pair(conv_fprop_kernel<0, true>, dim3(grid2), dim3(kFpropThreads), smem_bytes, stream, p));
    GAP_CUDA(cudaGetLastError());
    return 0;
  }
  const int grid = balanced(p.total_tiles, sms);
  if (bwd)
    GAP_CUDA(launch_pdl(conv_fprop_kernel<1>, dim3(grid), dim3(kFpropThreads), smem_bytes, stream, p));
  else if (p.accum)
    GAP_CUDA(launch_pdl(conv_fprop_kernel<2>, dim3(grid), dim3(kFpropThreads), smem_bytes, stream, p));
  else
    GAP_CUDA(launch_pdl(conv_fprop_kernel<0>, dim3(grid), dim3(kFpropThreads), smem_bytes, stream, p));
  GAP_CUDA(cudaGetLastError());
  return 0;
}
