// gemm_tc.cu -- tcgen05 / TMEM implicit-GEMM kernel fed by TMA (sm_100a).
//
// One persistent, warp-specialised kernel computes  D[rows, cols] = sum over "K blocks" of A_box * B_box^T  with bf16
// operands and fp32 accumulation in tensor memory.  A "K block" is 64 channels of one filter tap: the activation
// operand of tap (ky, kx) is simply the NHWC tensor box shifted by (ky-1, kx-1), fetched by a 4-D TMA box load whose
// out-of-bounds elements are zero-filled by the hardware -- that IS the convolution's zero padding, so no im2col buffer
// exists anywhere.  The same kernel runs 3x3 / 1x1 convolutions, stride-2 convolutions (four phase-subsampled tensor
// maps), nearest-x2-upsample + 3x3 (one launch per output phase), a fused second K segment (the ResnetBlock 1x1
// `res_conv`), and the batched attention products Q*K^T and P*V.
//
// Warp roles (320 threads): warps 0-7 = epilogue, warp 8 = TMA producer, warp 9 = TMEM allocator + single-thread
// tcgen05.mma issuer (tcgen05.ld -> bias / time-embedding / activation / residual -> global).  Two accumulator
// buffers in TMEM let the epilogue of tile i overlap the MMAs of tile i+1.
//
// Variants (template parameters): HALO / ROWS (tiles that are segments of image rows: one halo tile serves the 9 taps), VM (vertical tap
// merge for 64-column tiles), FUSE (GroupNorm + Swish of the INPUT applied between TMA and MMA by extra transform warps), STG (epilogue
// stores staged through shared memory), SPLIT (the K loop of a tile cut over the CTAs of a thread-block cluster, fp32 partials exchanged
// through distributed shared memory) and PAIR (cta_group::2: two CTAs of one TPC share a 256 x 256 tile, each staging its own 128 rows of
// activations and half of the weight columns; the leader issues the MMAs and commits to the barriers of both).
//
// Reference call sites replaced: every nn.Conv2d on the UNet path (nn_modules/resnet.py:24,51,78-79,
// functional_layers.py:64,79, resdiff/unet.py:68, guided_cross_attention.py:20-22) and the attention einsums
// (nn_modules/resnet.py:90-97, guided_cross_attention.py:34-41).
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "tc_common.cuh"

namespace wsr {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                       // bf16 elements = 128 bytes = one swizzle row
constexpr int kABytes = kBlockM * kBlockK * 2;    // 16 KB
constexpr int kMaxEntries = 18;              // 16 taps (WSR_MAX_TAPS) + fused 1x1 segment + spare
constexpr int kNumAMaps = 5;
constexpr int kNumBMaps = 3;                     // [0] conv weights, [1] fused 1x1 segment, [2] vertically merged taps

struct TcEntry {
  int16_t amap, bmap;      // tensor-map indices
  int16_t a_c0;            // first channel coordinate in A
  int16_t d1, d2;          // coordinate offsets in A dims 1, 2 (w, h)
  int16_t b_k0;            // first k coordinate in B
  int16_t b_z;             // B coordinate 2 (filter tap)
  int16_t nchunks;         // number of 64-channel K blocks
};

struct TcParams {
  CUtensorMap amap[kNumAMaps];
  CUtensorMap bmap[kNumBMaps];
  TcEntry e[kMaxEntries];
  int n_entries;
  int total_kb;                 // sum of nchunks
  int t1, t2, t3;               // A box extents along dims 1..3; rows_box = t1*t2*t3 <= 128
  int g1, g2, g3;               // tiles along dims 1..3
  int nbatch;                   // extra batch dimension (attention GEMMs); 1 for convolutions
  int a_zmul, b_zmul;           // A coord3 += zb*a_zmul ; B coord2 += zb*b_zmul
  int n_tiles;                  // tiles along columns
  int a_bytes;                  // bytes one A tile load delivers (rows_box * 128, or 8 KB per 64-row block when MN-major)
  int b_bytes;                  // bytes one B tile load delivers; 0 = BLOCK_N * 128 (K-major box)
  int a_mn, b_mn;               // operand is MN-major (contiguous along rows / columns, strided along K): loaded as
                                // [64 MN][64 K] boxes 8 KB apart and consumed through the MN-major UMMA descriptor
  int a_blk, b_blk;             // number of such 64-wide boxes per tile
  int halo_rows;                // halo mode: output rows per tile (1 or 2; 2 = two accumulators share every weight tile)
  int n_taps, halo_bytes;       // halo mode: e[0..n_taps) are filter taps served from one (t1+2) x 3 halo tile per chunk
  int M1, M2, M3;               // valid row extents (masking)
  int Ncols;                    // valid columns
  void* out; int out_dtype;
  long long o_s1, o_s2, o_s3, o_sb, o_sc;
  int mul1, off1, mul2, off2;   // output coordinate = i*mul + off along dims 1, 2
  const float* bias;
  const float* rowvec; int rowvec_ld;
  int act; float out_scale;
  const void* res; int res_dtype; long long r_s1, r_s2, r_s3, r_sb, r_sc; float res_scale;
  const void* res2; int res2_dtype; long long q_s1, q_s2, q_s3, q_sb, q_sc; float res2_scale;
  double* stats; int stats_ld;  // fused GroupNorm statistics of the output (needs t1*t2 % 32 == 0), or nullptr
  // fused GroupNorm (+ Swish) of the INPUT (halo mode, FUSE kernels): the activation operand is not fetched by TMA but by
  // four "transform" warps that read the raw tensor from global memory, apply a = act(x * scale[n][c] + shift[n][c]) and
  // write the 128B-swizzled tile themselves (out-of-image pixels stay zero = the convolution's padding of the
  // NORMALISED tensor).  gn_tab: [N][gn_ld] float2 (scale, shift) from wsr_gn_finalize.
  // split-K (SPLIT kernels, classic mode, one work item per CTA): the K blocks of a tile are cut into `ksplit` contiguous ranges of
  // `kb_split` blocks; the `ksplit` CTAs of a tile form a thread-block CLUSTER, CTA s accumulates range s in its own tensor memory, then
  // the partial tiles are exchanged through distributed shared memory: CTA s finishes the 32-column chunks ch with ch % ksplit == s and
  // receives the other CTAs' partials of those chunks in its (by then idle) operand ring.
  int ksplit, kb_split;
  int pair;                     // classic mode, N = 256: run as CTA pairs (PAIR kernels); the weight map's box is then 128 rows
  const void* xg; int xg_ld, xg_H, xg_W;
  const void* x2g; int x2g_ld;
  const float2* gn_tab; int gn_ld; int gn_act;
};

constexpr int kEpiWarps = 8;                      // two warps per TMEM lane quadrant, each owning half of the columns
// Fused-GroupNorm kernels: 20 warps = 5 warpgroups.  Warpgroups 0-1 = the 8 epilogue warps, warpgroup 2 = TMA producer (warp 8), MMA
// issuer (warp 9) and two idle warps, warpgroups 3-4 = 8 transform warps.  All warps of a kernel start with the same register
// count (65536 / 640 -> 96), which neither fits the 168-register staged epilogue nor is needed by the single-thread roles, so the
// warpgroups re-balance with setmaxnreg at the top of their role branches: 168 / 40 / 48 registers.  The increase can only be served
// from registers the CTA itself gives back, so the budget is the LAUNCH allocation, not the register file:
// 256*168 + 128*40 + 256*48 = 60416 <= 640 * 96 = 61440 (a plan that sums to more than the launch allocation deadlocks in the
// setmaxnreg.inc of the epilogue warps).
// Round 1 ran 4 transform warps at the common 128-register cap: one warp per scheduler could not hide its own latencies
// (0.30 ms for the transform alone on the 64->64 @128x256 layer) and the epilogue spilled.
constexpr int kXfWarps = 8;                       // transform warps of the fused-GroupNorm kernels
constexpr int kXfFirstWarp = 12;
constexpr int kTcThreads = 64 + 32 * kEpiWarps;
constexpr int kTcThreadsFused = 32 * (kXfFirstWarp + kXfWarps);   // 640
// halo tile of ROWS output rows: (ROWS + 2) x 130 pixels x 128 bytes, rounded up to a multiple of 1024
constexpr int halo_stage_bytes(int rows) { return ((rows + 2) * 130 * 128 + 1023) / 1024 * 1024; }

constexpr int next_pow2(int v) { int p = 32; while (p < v) p *= 2; return p; }

// VM ("vertical tap merge", halo mode, N = 64): a halo row feeds the three output rows above / at / below it through
// the taps dy = +1, 0, -1.  With the accumulators of consecutive output rows laid out side by side in TMEM, ONE MMA per
// (halo row, dx) with the weight matrices [dy=+1 | dy=0 | dy=-1] stacked along N (192 columns) updates all three: the
// 128-pixel activation operand -- whose shared-memory fetch bounds the N = 64 layers -- is read 5 times per 3 output
// rows instead of 9 times.
// PAIR (classic mode, N = 256): two CTAs on one TPC share a 256 x 256 tile through cta_group::2 MMAs -- each CTA stages its own 128 rows
// of A and only HALF of the B columns, so a K block costs 32 KB of L2 -> SM traffic per SM instead of 48 KB.  At ~70 bytes per clock
// and SM that is the difference between 690 and 460 cycles against 512 cycles of MMA: the single-CTA kernel is fetch-bound (ncu: tensor
// pipe 61 % busy on the 32x64 / 16x32 / 8x16 levels), the pair is not.
template <int BLOCK_N, bool HALO, int ROWS, bool VM = false, bool PAIR = false> struct TcCfg {
  static constexpr int kHaloStage = halo_stage_bytes(ROWS);
  static constexpr int kBTile = (PAIR ? BLOCK_N / 2 : BLOCK_N) * kBlockK * 2;   // one weight tile (PAIR: this CTA's half of the columns)
  static constexpr int kBBytes = VM ? 3 * kBTile : kBTile;             // one stage of the weight ring
  // classic mode: one ring of {A tile, B tile} stages.  halo mode: a ring of activation halo tiles (one per 64-channel
  // chunk, shared by the 9 taps) and a separate ring of weight tiles.
  static constexpr int kStages = PAIR ? 6 : (BLOCK_N >= 256 ? 4 : (BLOCK_N >= 128 ? 6 : 8));
  static constexpr int kAStages = 2;
  static constexpr int kBStages = VM ? 2 : (BLOCK_N >= 256 ? 3 : (BLOCK_N >= 128 ? (ROWS > 1 ? 4 : 6) : (ROWS >= 4 ? 3 : 8)));
  static constexpr int kSmemData = HALO ? kAStages * kHaloStage + kBStages * kBBytes : kStages * (kABytes + kBBytes);
  static constexpr int kAccCols = ROWS * BLOCK_N;                           // one accumulator set (ROWS output rows)
  static constexpr int kTmemCols = next_pow2(2 * kAccCols);                // power of two for 32..512
  static_assert(kTmemCols <= 512, "TMEM budget");
  static constexpr int kBsumBytes = HALO ? 16 * BLOCK_N : 0;                // per epilogue warp: bias + time-embedding row of its columns
  // per epilogue warp: a 16-row x 64-byte staging buffer through which residual loads and output stores are re-shaped from
  // "one row per lane" (32 different 128-byte lines per instruction) to "four lanes per row" (8 lines per instruction);
  // the ROWS = 4 configuration has no shared memory left for it
  static constexpr int kStgBytes = (HALO && ROWS >= 4) ? 0 : 8 * 1024;
  static constexpr int kSmemBytes = kSmemData + 1024 /*align slack*/ + 512 /*barriers*/ + kBsumBytes + kStgBytes;
  static_assert(kSmemBytes <= 232448, "shared memory budget");
  // instruction descriptor: D=f32, A=B=bf16, both K-major, N, M=128 (256 across a CTA pair)
  static constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)((PAIR ? 2 : 1) * kBlockM >> 4) << 24);
};

struct TileCoord { int nt, i1, i2, i3, zb; };

__device__ __forceinline__ TileCoord decode_tile(const TcParams& p, int tile) {
  TileCoord t;
  t.nt = tile % p.n_tiles;
  int mt = tile / p.n_tiles;
  t.i1 = mt % p.g1; mt /= p.g1;
  t.i2 = mt % p.g2; mt /= p.g2;
  t.i3 = mt % p.g3;
  t.zb = mt / p.g3;
  return t;
}

// ------------------------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------------------------
template <int BLOCK_N, bool HALO, int ROWS, bool FUSE = false, bool VM = false, bool STG = false, bool SPLIT = false, bool PAIR = false>
__global__ void __launch_bounds__(FUSE ? kTcThreadsFused : kTcThreads, 1) gemm_tc_kernel(const __grid_constant__ TcParams p) {
  static_assert(!SPLIT || (!HALO && STG), "split-K: classic tiles with the staged epilogue only");
  static_assert(!PAIR || (!HALO && !SPLIT && !FUSE && BLOCK_N == 256), "CTA pairs: classic 256-column tiles only");
  // STG: the epilogue moves residual loads and output stores through a per-warp shared-memory staging buffer (see TcCfg::kStgBytes);
  // the host selects it only when stage_preconditions() hold (bf16 output / residual, unit channel stride, 16-byte aligned rows)
  // register budget: 10 warps = 3 warps on the fullest scheduler, 16384 / 3 / 32 -> 168 registers per thread at most
  static_assert(256 * 168 + 128 * 40 + 256 * 48 <= kTcThreadsFused * 96, "setmaxnreg plan exceeds the launch allocation");
  static_assert(!FUSE || HALO, "the fused-GroupNorm input path exists in halo mode only");
  static_assert(!VM || (HALO && BLOCK_N == 64), "vertical tap merge: halo mode, N = 64");
  using Cfg = TcCfg<BLOCK_N, HALO, ROWS, VM, PAIR>;
  static_assert(!STG || Cfg::kStgBytes > 0, "no staging buffer in this configuration");
  constexpr int kHaloStage = Cfg::kHaloStage;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + Cfg::kSmemData);
  // classic: full[kStages], empty[kStages] | halo: fullA[2], emptyA[2], fullB[kBStages], emptyB[kBStages]
  constexpr int kRingA = HALO ? Cfg::kAStages : Cfg::kStages;
  constexpr int kRingB = HALO ? Cfg::kBStages : 0;
  uint64_t* full_a = bars;
  uint64_t* empty_a = full_a + kRingA;
  uint64_t* full_b = empty_a + kRingA;
  uint64_t* empty_b = full_b + kRingB;
  uint64_t* tfull_bar = empty_b + kRingB;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* full_raw = tempty_bar + 2;                       // FUSE: TMA landed the raw tile (transform warps wait on it)
  // FUSE, halo chunks: the stage is handed over ROW BY ROW -- row_raw[stage][h]: halo row h has landed (one TMA box per row);
  // row_rdy[stage][h]: the transform warps have rewritten it.  With whole-stage barriers a stage went load -> transform -> MMA
  // strictly one after the other (~5 + 2.4 + 3.5 us per 83 KB stage of the 64->64 layer), and two stages cannot hide three serial
  // phases: the fused layer ran at the speed of conv + separate GroupNorm pass.  Row by row the three phases overlap inside a stage.
  constexpr int kRowMax = 6;
  uint64_t* row_raw = full_raw + 2;                          // [2][kRowMax]
  uint64_t* row_rdy = row_raw + 2 * kRowMax;                 // [2][kRowMax]
  // SPLIT: done_bar -- every CTA of the cluster has finished its K range (its operand ring may be overwritten); recv_bar -- every other
  // CTA has delivered its partials of this CTA's chunks
  uint64_t* done_bar = row_rdy + 2 * kRowMax;
  uint64_t* recv_bar = done_bar + 1;
  uint32_t* tmem_slot = (uint32_t*)(recv_bar + 1);
  static_assert(!FUSE || ROWS + 2 <= kRowMax, "row barriers");
  uint8_t* smem_b = smem + Cfg::kAStages * kHaloStage;      // halo mode only

  // warp roles: 0..7 epilogue, 8 TMA producer, 9 MMA issuer.  The issue arbiter favours the HIGHEST warp id on an SMSP, so
  // the two latency-critical single-thread roles get the top ids and are never starved by the epilogue warps.
  // fused kernels: warps 10..13 are the transform warps.  They get the TOP ids: while they work the producer / MMA threads
  // mostly spin on barriers, and a spinning higher-priority warp on the same scheduler starved them (4x slower transform).
  constexpr int kProducerWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;
  constexpr int kXfWarp0 = kXfFirstWarp;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.g1 * p.g2 * p.g3 * p.nbatch * p.n_tiles;
  // contiguous tile range per CTA: consecutive tiles share the image (register-accumulated GroupNorm statistics) and
  // neighbouring rows (halo re-reads hit L2)
  // SPLIT: the grid is exactly (tiles x ksplit) CTAs, CTA = (tile, split)
  const int split_s = SPLIT ? (int)blockIdx.x % p.ksplit : 0;
  // PAIR: the grid is a row of 2-CTA clusters; a pair walks "pair tiles" tq = (row-tile pair, column tile) and CTA `rank` of the pair
  // owns row tile 2 * pair + rank of each (the host guarantees an even number of row tiles)
  const int pair_rank = PAIR ? (int)cluster_ctarank() : 0;
  const int n_work = PAIR ? total_tiles / 2 : total_tiles;
  const int n_cta = PAIR ? (int)gridDim.x / 2 : (int)gridDim.x;
  const int cta_i = PAIR ? (int)blockIdx.x / 2 : (int)blockIdx.x;
  const int tile_begin = SPLIT ? (int)blockIdx.x / p.ksplit : (int)((long long)cta_i * n_work / n_cta);
  const int tile_end = SPLIT ? tile_begin + 1 : (int)((long long)(cta_i + 1) * n_work / n_cta);
  auto work_tile = [&](int tq) { return PAIR ? ((tq / p.n_tiles) * 2 + pair_rank) * p.n_tiles + tq % p.n_tiles : tq; };
  const int kb0 = SPLIT ? split_s * p.kb_split : 0;
  const int kb1 = SPLIT ? min(p.total_kb, kb0 + p.kb_split) : p.total_kb;

  if (warp == kProducerWarp && lane == 0) {
    for (int i = 0; i < kNumAMaps; ++i) prefetch_tmap(&p.amap[i]);
    for (int i = 0; i < kNumBMaps; ++i) prefetch_tmap(&p.bmap[i]);
    for (int s = 0; s < kRingA; ++s) { mbar_init(&full_a[s], FUSE ? kXfWarps : 1); mbar_init(&empty_a[s], 1); }
    for (int s = 0; s < kRingB; ++s) { mbar_init(&full_b[s], 1); mbar_init(&empty_b[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], (PAIR ? 2 : 1) * kEpiWarps); mbar_init(&full_raw[a], 1); }
    if constexpr (FUSE) {
      for (int i = 0; i < 2 * kRowMax; ++i) { mbar_init(&row_raw[i], 1); mbar_init(&row_rdy[i], kXfWarps); }
    }
    if constexpr (SPLIT) { mbar_init(done_bar, (uint32_t)p.ksplit); mbar_init(recv_bar, (uint32_t)((p.ksplit - 1) * kEpiWarps)); }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == kMmaWarp) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  // PAIR: the peer must not signal this CTA's barriers (TMA transaction bytes, MMA commits, accumulator hand-back) before they exist
  if constexpr (PAIR || SPLIT) cluster_sync_all(); else __syncthreads();      // SPLIT: peers arrive on done_bar / recv_bar and write into the ring
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // FUSE: register re-balancing between the warpgroups (see kXfWarps) -- the setmaxnreg of each role is the FIRST statement of its
  // branch below, so that the compiler sees which budget governs which code (every warp of a warpgroup executes the same value)
  // programmatic dependent launch: everything above touched only this CTA's shared / tensor memory and the (kernel-parameter)
  // tensor maps; from here on the kernel reads what earlier launches produced and overwrites what they may still be reading
  pdl_launch_dependents();
  pdl_wait();

  if (warp == kProducerWarp) {
    // ===================== TMA producer =====================
    if constexpr (FUSE) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (lane == 0) {
      int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
      for (int tq = tile_begin; tq < tile_end; ++tq) {
        const int tile = work_tile(tq);
        const TileCoord t = decode_tile(p, tile);
        const int c1 = t.i1 * p.t1, c2 = t.i2 * (HALO ? ROWS : p.t2), c3 = t.i3 * p.t3 + t.zb * p.a_zmul;
        if constexpr (!HALO) {
          int kbi = 0;
          for (int ei = 0; ei < p.n_entries; ++ei) {
            const TcEntry e = p.e[ei];
            for (int c = 0; c < e.nchunks; ++c, ++kbi) {
              if constexpr (SPLIT) { if (kbi < kb0 || kbi >= kb1) continue; }
              mbar_wait(&empty_a[sa], pa ^ 1);
              uint8_t* st = smem + sa * (kABytes + Cfg::kBBytes);
              if constexpr (PAIR) {
                // both CTAs' loads complete on the leader's barrier (the leader's MMA thread is the only consumer)
                if (pair_rank == 0) mbar_expect_tx(&full_a[sa], (uint32_t)(2 * (p.a_bytes + Cfg::kBBytes)));
                tma_load_4d_pair(st, &p.amap[e.amap], &full_a[sa], e.a_c0 + c * kBlockK, c1 + e.d1, c2 + e.d2, c3);
                tma_load_3d_pair(st + kABytes, &p.bmap[e.bmap], &full_a[sa], e.b_k0 + c * kBlockK, t.nt * BLOCK_N + pair_rank * (BLOCK_N / 2), e.b_z);
                if (++sa == kRingA) { sa = 0; pa ^= 1; }
                continue;
              }
              mbar_expect_tx(&full_a[sa], (uint32_t)(p.a_bytes + (p.b_bytes ? p.b_bytes : Cfg::kBBytes)));
              if (!p.a_mn) {
                tma_load_4d(st, &p.amap[e.amap], &full_a[sa], e.a_c0 + c * kBlockK, c1 + e.d1, c2 + e.d2, c3);
              } else {
                for (int j = 0; j < p.a_blk; ++j) tma_load_4d(st + j * 8192, &p.amap[e.amap], &full_a[sa], c1 + 64 * j, e.a_c0 + c * kBlockK, 0, c3);
              }
              if (!p.b_mn) {
                tma_load_3d(st + kABytes, &p.bmap[e.bmap], &full_a[sa], e.b_k0 + c * kBlockK, t.nt * BLOCK_N, e.b_z + t.zb * p.b_zmul);
              } else {
                for (int j = 0; j < p.b_blk; ++j)
                  tma_load_3d(st + kABytes + j * 8192, &p.bmap[e.bmap], &full_a[sa], t.nt * BLOCK_N + 64 * j, e.b_k0 + c * kBlockK, e.b_z + t.zb * p.b_zmul);
              }
              if (++sa == kRingA) { sa = 0; pa ^= 1; }
            }
          }
        } else {
          // taps e[0 .. n_taps): one halo tile per 64-channel chunk, then one weight tile per tap
          const int nch = p.e[0].nchunks;
          for (int c = 0; c < nch; ++c) {
            {
              mbar_wait(&empty_a[sa], pa ^ 1);
              if constexpr (FUSE) {
                // one box per halo row (amap[1]: the same tensor, box = one row of t1 + 2 pixels), each on its own barrier
                const int row_bytes = (p.t1 + 2) * 128;
                for (int h = 0; h < ROWS + 2; ++h) {
                  mbar_expect_tx(&row_raw[sa * kRowMax + h], (uint32_t)row_bytes);
                  tma_load_4d(smem + sa * kHaloStage + h * row_bytes, &p.amap[1], &row_raw[sa * kRowMax + h], c * kBlockK, c1 - 1, c2 - 1 + h, c3);
                }
              } else {
                mbar_expect_tx(&full_a[sa], (uint32_t)p.halo_bytes);
                tma_load_4d(smem + sa * kHaloStage, &p.amap[p.e[0].amap], &full_a[sa], c * kBlockK, c1 - 1, c2 - 1, c3);
              }
              if constexpr (FUSE) {
                // the box that will land in this stage the NEXT time round (two halo loads ahead) goes to L2 now: with the transform
                // between load and MMA a stage is refilled only after load + transform + MMA of its previous content, so the refill
                // latency is on the critical path and should be an L2 hit, not an HBM round trip
                const int idx = c + kRingA;
                const int t2i = tile + idx / nch, c2i = idx % nch;
                if (t2i < tile_end) {
                  const TileCoord u = decode_tile(p, t2i);
                  tma_prefetch_4d(&p.amap[p.e[0].amap], c2i * kBlockK, u.i1 * p.t1 - 1, u.i2 * ROWS - 1, u.i3 * p.t3 + u.zb * p.a_zmul);
                }
              }
              if (++sa == kRingA) { sa = 0; pa ^= 1; }
            }
            if constexpr (VM) {
              // one [3 x 64 rows] box per horizontal offset dx: rows = weights of dy = +1, 0, -1 (wsr vmerge pack)
              for (int dxi = 0; dxi < 3; ++dxi) {
                mbar_wait(&empty_b[sb], pb ^ 1);
                mbar_expect_tx(&full_b[sb], (uint32_t)Cfg::kBBytes);
                tma_load_3d(smem_b + sb * Cfg::kBBytes, &p.bmap[2], &full_b[sb], c * kBlockK, 0, dxi);
                if (++sb == kRingB) { sb = 0; pb ^= 1; }
              }
            } else {
            for (int ei = 0; ei < p.n_taps; ++ei) {
              const TcEntry e = p.e[ei];
              mbar_wait(&empty_b[sb], pb ^ 1);
              mbar_expect_tx(&full_b[sb], (uint32_t)Cfg::kBBytes);
              tma_load_3d(smem_b + sb * Cfg::kBBytes, &p.bmap[e.bmap], &full_b[sb], e.b_k0 + c * kBlockK, t.nt * BLOCK_N, e.b_z);
              if (++sb == kRingB) { sb = 0; pb ^= 1; }
            }
            }
          }
          // remaining entries (fused 1x1 segment): plain 128-row activation tiles in the same A ring
          for (int ei = p.n_taps; ei < p.n_entries; ++ei) {
            const TcEntry e = p.e[ei];
            for (int c = 0; c < e.nchunks; ++c) {
              {
                uint64_t* fb = FUSE ? &full_raw[sa] : &full_a[sa];
                mbar_wait(&empty_a[sa], pa ^ 1);
                mbar_expect_tx(fb, (uint32_t)p.a_bytes);
                tma_load_4d(smem + sa * kHaloStage, &p.amap[e.amap], fb, e.a_c0 + c * kBlockK, c1 + e.d1, c2 + e.d2, c3);
                if (++sa == kRingA) { sa = 0; pa ^= 1; }
              }
              mbar_wait(&empty_b[sb], pb ^ 1);
              mbar_expect_tx(&full_b[sb], (uint32_t)Cfg::kBTile);
              tma_load_3d(smem_b + sb * Cfg::kBBytes, &p.bmap[e.bmap], &full_b[sb], e.b_k0 + c * kBlockK, t.nt * BLOCK_N, e.b_z);
              if (++sb == kRingB) { sb = 0; pb ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer =====================
    if constexpr (FUSE) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (lane == 0) {
      int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
      uint32_t ph_row = 0u, ph_x2 = 0u;     // FUSE: per-stage phase bits (bit = stage) of the row barriers / of full_a (x2 uses)
      int it = 0;
      for (int tile = tile_begin; tile < ((PAIR && pair_rank != 0) ? tile_begin : tile_end); ++tile, ++it) {   // PAIR: the leader issues for both
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * Cfg::kAccCols);
        if constexpr (!HALO) {
          // K-major operand: +32 bytes along K inside the swizzle atom = +2 in the address field, LBO unused (1).
          // MN-major operand: 16 K rows of 128 bytes = +128, LBO = 8 KB (the next 64-wide box).
          const uint32_t a_st = p.a_mn ? 128u : 2u, b_st = p.b_mn ? 128u : 2u;
          const uint32_t a_lbo = (p.a_mn ? (8192u >> 4) : 1u) << 16, b_lbo = (p.b_mn ? (8192u >> 4) : 1u) << 16;
          const uint32_t idesc = Cfg::kIdesc | ((uint32_t)p.a_mn << 15) | ((uint32_t)p.b_mn << 16);
          for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(&full_a[sa], pa);
            tc_fence_after();
            const uint32_t s_lo = (smem_u32(smem + sa * (kABytes + Cfg::kBBytes)) & 0x3FFFFu) >> 4;
            const uint32_t a_lo = s_lo | a_lbo;
            const uint32_t b_lo = (s_lo + (uint32_t)(kABytes >> 4)) | b_lbo;
            if constexpr (PAIR) {
              umma_bf16_lo_pair(d_tmem, a_lo, b_lo, idesc, kb != kb0 ? 1u : 0u);
              umma_bf16_lo_pair(d_tmem, a_lo + 2u, b_lo + 2u, idesc, 1u);
              umma_bf16_lo_pair(d_tmem, a_lo + 4u, b_lo + 4u, idesc, 1u);
              umma_bf16_lo_pair(d_tmem, a_lo + 6u, b_lo + 6u, idesc, 1u);
              umma_commit_pair(&empty_a[sa]);                           // frees the stage in both CTAs
              if (kb == kb1 - 1) umma_commit_pair(&tfull_bar[acc]);     // both epilogues
            } else {
            umma_bf16_lo(d_tmem, a_lo, b_lo, idesc, kb != kb0 ? 1u : 0u);
            umma_bf16_lo(d_tmem, a_lo + a_st, b_lo + b_st, idesc, 1u);
            umma_bf16_lo(d_tmem, a_lo + 2 * a_st, b_lo + 2 * b_st, idesc, 1u);
            umma_bf16_lo(d_tmem, a_lo + 3 * a_st, b_lo + 3 * b_st, idesc, 1u);
            umma_commit(&empty_a[sa]);
            if (kb == kb1 - 1) umma_commit(&tfull_bar[acc]);
            }
            if (++sa == kRingA) { sa = 0; pa ^= 1; }
          }
        } else {
          int kb = 0;
          const int nch = p.e[0].nchunks;
          const int pitch = p.t1 + 2;
          for (int c = 0; c < nch; ++c) {
            // FUSE: rows become readable one by one (row_rdy); `rows_ok` = halo rows of this stage already waited for
            int rows_ok = 0;
            auto need_rows = [&](int upto) {          // make halo rows [0, upto) of the current stage readable
              if constexpr (FUSE) {
                if (rows_ok < upto) {
                  for (; rows_ok < upto; ++rows_ok) mbar_wait(&row_rdy[sa * kRowMax + rows_ok], (ph_row >> sa) & 1u);
                  tc_fence_after();
                }
              }
            };
            if constexpr (!FUSE) mbar_wait(&full_a[sa], pa);
            const uint32_t a_lo0 = desc_lo(smem_u32(smem + sa * kHaloStage));
            const uint32_t pitch8 = (uint32_t)pitch * 8u;
            if constexpr (VM) {
              constexpr uint32_t kIdBase = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBlockM >> 4) << 24);
              for (int dxi = 0; dxi < 3; ++dxi, ++kb) {
                mbar_wait(&full_b[sb], pb);
                tc_fence_after();
                const uint32_t v_lo = a_lo0 + (uint32_t)dxi * 8u;                 // halo column offset dx + 1 = dxi
                const uint32_t b_lo = desc_lo(smem_u32(smem_b + sb * Cfg::kBBytes));
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                  if (kb == 0 && k == 0) {
                    // very first K step of the tile: every accumulator block starts from zero, which a merged MMA cannot
                    // express (one accumulate flag per instruction) -> nine plain N = 64 MMAs, first touch overwrites
                    // (issued in halo-row order so that the fused-GroupNorm kernels can start as soon as row 0 is transformed; output
                    // row rr is still first touched by its dy = -1 tap, halo row rr)
#pragma unroll
                    for (int hr = 0; hr < ROWS + 2; ++hr) {
                      need_rows(hr + 1);
#pragma unroll
                      for (int dyi = 0; dyi < 3; ++dyi) {      // dy = dyi - 1 reads halo row rr + dyi; weights block 2 - dyi
                        const int rr = hr - dyi;
                        if (rr >= 0 && rr < ROWS)
                          umma_bf16_lo(d_tmem + (uint32_t)(rr * 64), v_lo + (uint32_t)hr * pitch8, b_lo + (uint32_t)(2 - dyi) * 512u,
                                       kIdBase | (8u << 17), dyi != 0 ? 1u : 0u);
                      }
                    }
                  } else {
#pragma unroll
                    for (int hr = 0; hr < ROWS + 2; ++hr) {
                      need_rows(hr + 1);
                      // halo row hr feeds output rows hr-2 (dy=+1, block 0), hr-1 (dy=0, block 1), hr (dy=-1, block 2)
                      const int r_lo = hr - 2 < 0 ? 0 : hr - 2, r_hi = hr < ROWS - 1 ? hr : ROWS - 1;
                      const int nblk = r_hi - r_lo + 1, blk0 = r_lo - (hr - 2);
                      umma_bf16_lo(d_tmem + (uint32_t)(r_lo * 64), v_lo + (uint32_t)hr * pitch8 + (uint32_t)(2 * k),
                                   b_lo + (uint32_t)blk0 * 512u + (uint32_t)(2 * k), kIdBase | ((uint32_t)(nblk * 8) << 17), 1u);
                    }
                  }
                }
                umma_commit(&empty_b[sb]);
                if (++sb == kRingB) { sb = 0; pb ^= 1; }
              }
            } else {
            for (int ei = 0; ei < p.n_taps; ++ei, ++kb) {
              const TcEntry e = p.e[ei];
              mbar_wait(&full_b[sb], pb);
              tc_fence_after();
              // tap (dy, dx) = the 128 consecutive halo rows starting at row (dy+1)*pitch + (dx+1).  The 128B swizzle is a
              // function of the absolute shared-memory address bits (the halo buffer is 1024-byte aligned, so the
              // descriptor's base-offset field stays 0), exactly as for the +32-byte K advance below.
              const uint32_t t_lo = a_lo0 + (uint32_t)((e.d2 + 1) * pitch + (e.d1 + 1)) * 8u;    // 128-byte rows = 8 address units
              const uint32_t b_lo = desc_lo(smem_u32(smem_b + sb * Cfg::kBBytes));
              need_rows(e.d2 + 1 + ROWS);                  // this tap reads halo rows dy + 1 .. dy + ROWS
              // k outer, row inner: consecutive MMAs accumulate into different TMEM tiles
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k) {
#pragma unroll
                for (int rr = 0; rr < ROWS; ++rr)       // output row rr of the tile reads halo rows rr .. rr+2
                  umma_bf16_lo(d_tmem + (uint32_t)(rr * BLOCK_N), t_lo + (uint32_t)rr * pitch8 + (uint32_t)(2 * k), b_lo + (uint32_t)(2 * k),
                               Cfg::kIdesc, k != 0 ? 1u : (kb != 0 ? 1u : 0u));
              }
              umma_commit(&empty_b[sb]);
              if (++sb == kRingB) { sb = 0; pb ^= 1; }
            }
            }
            need_rows(ROWS + 2);                           // (every row barrier of the stage has been consumed: phases stay in step)
            umma_commit(&empty_a[sa]);
            if constexpr (FUSE) ph_row ^= 1u << sa;
            if (++sa == kRingA) { sa = 0; pa ^= 1; }
          }
          for (int ei = p.n_taps; ei < p.n_entries; ++ei) {
            const int n2 = p.e[ei].nchunks;
            for (int c = 0; c < n2; ++c, ++kb) {
              if constexpr (FUSE) { mbar_wait(&full_a[sa], (ph_x2 >> sa) & 1u); ph_x2 ^= 1u << sa; }
              else mbar_wait(&full_a[sa], pa);
              mbar_wait(&full_b[sb], pb);
              tc_fence_after();
              const uint32_t a_lo = desc_lo(smem_u32(smem + sa * kHaloStage));
              const uint32_t b_lo = desc_lo(smem_u32(smem_b + sb * Cfg::kBBytes));
              const uint32_t slab8 = (uint32_t)p.t1 * 8u;      // plain tile: ROWS consecutive slabs of t1 pixel rows
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k) {
#pragma unroll
                for (int rr = 0; rr < ROWS; ++rr)
                  umma_bf16_lo(d_tmem + (uint32_t)(rr * BLOCK_N), a_lo + (uint32_t)rr * slab8 + (uint32_t)(2 * k), b_lo + (uint32_t)(2 * k),
                               Cfg::kIdesc, k != 0 ? 1u : (kb != 0 ? 1u : 0u));
              }
              umma_commit(&empty_b[sb]);
              umma_commit(&empty_a[sa]);
              if (++sb == kRingB) { sb = 0; pb ^= 1; }
              if (++sa == kRingA) { sa = 0; pa ^= 1; }
            }
          }
          umma_commit(&tfull_bar[acc]);
        }
      }
    }
  } else if (FUSE && warp > kMmaWarp && warp < kXfWarp0) {
    // the two spare warps of the producer / MMA warpgroup: give their registers back and leave
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
  } else if (FUSE && warp >= kXfWarp0 && warp < kXfWarp0 + kXfWarps) {
    // ===================== transform warps (fused GroupNorm + activation of the input) =====================
    // The raw halo tile has been landed by TMA (zero-filled outside the image); each thread rewrites IN PLACE the 16-byte
    // vectors of one logical channel column: a = act(x * scale + shift), leaving out-of-image pixels at zero (the padding
    // applies to the normalised tensor), then releases the stage to the MMA issuer.  (Fetching the tile with ordinary
    // loads instead was 4x slower: with 227 KB of shared memory carved out, L1 has almost no lines left for misses in flight.)
    if constexpr (FUSE) {
      asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
      const int xt = threadIdx.x - 32 * kXfWarp0;           // 0 .. 32 * kXfWarps - 1
      const int j = xt & 7;                                 // logical 16-byte column (8 channels) owned by this thread
      const int slot = xt >> 3;                             // pixel slot inside a halo row; pixels advance by kXfSlots
      constexpr int kXfSlots = 4 * kXfWarps;                // 32
      constexpr int U = 3;                                  // loads in flight per thread; 2 x 3 passes cover a halo row of up to 192 pixels
      const int pitch = p.t1 + 2;
      int sa = 0; uint32_t pa = 0;
      uint32_t ph_row = 0u, ph_x2 = 0u;                     // per-stage phase bits (bit = stage)
      const bool swish = p.gn_act == WSR_ACT_SWISH;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        const TileCoord t = decode_tile(p, tile);
        const int c1 = t.i1 * p.t1, c2 = t.i2 * ROWS, c3 = t.i3;
        const int nch = p.e[0].nchunks;
        // valid halo rows / columns of this tile (everything else is padding and stays zero)
        const int hy_lo = c2 - 1 < 0 ? 1 - c2 : 0, hy_hi = min(ROWS + 2, p.xg_H - (c2 - 1));
        const int hx_lo = c1 - 1 < 0 ? 1 - c1 : 0, hx_hi = min(pitch, p.xg_W - (c1 - 1));
        for (int c = 0; c < nch; ++c) {
          // PACKED bf16x2 arithmetic: a = fma(x, scale, shift), swish(a) = h * tanh(h) + h with h = a / 2 -- four FMA-pipe and one SFU
          // instruction per PAIR of channels.  The fp32 version of this loop (unpack, 2 FFMA, 2 x (FMUL, MUFU, FFMA), pack per pair;
          // ~100 instructions per 16-byte vector with the address / predicate code) ran at ~0.15 instructions per clock per warp: the
          // per-pair dependency chains did not fit the transform warps' 56 registers side by side, and the transform, not the tensor
          // pipe, set the pace of the fused layers (ncu: issue 40 %, tensor 17 %, SFU 15 %; profiles/r02_ncu_fused_gn_fp32_transform.txt).
          // Rounding: scale / shift and the intermediate a are rounded to bf16 (the unfused pass rounds only its output), i.e. about one
          // extra bf16 rounding per activation -- inside the 2e-2 budget of the bf16 mode (tests/test_parity_*_gpu.py run with the fusion).
          uint32_t sc2[4], sh2[4];
          {
            const float4* tp = (const float4*)(p.gn_tab + (long long)c3 * p.gn_ld + c * kBlockK + j * 8);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 v = __ldg(tp + q);                 // (scale, shift) of channels 2q, 2q + 1
              __nv_bfloat162 s2 = __floats2bfloat162_rn(v.x, v.z), h2 = __floats2bfloat162_rn(v.y, v.w);
              sc2[q] = *(uint32_t*)&s2; sh2[q] = *(uint32_t*)&h2;
            }
          }
          const uint32_t st_s = smem_u32(smem + sa * kHaloStage);
          for (int hy = 0; hy < ROWS + 2; ++hy) {
            // row by row: wait for this row's TMA box, rewrite it in place, hand it to the MMA issuer
            mbar_wait(&row_raw[sa * kRowMax + hy], (ph_row >> sa) & 1u);
            if (hy >= hy_lo && hy < hy_hi) {
#pragma unroll
             for (int u0 = 0; u0 < 6; u0 += U) {             // two batches of three passes: 96 + 96 pixel slots >= t1 + 2
              uint32_t raw[U][4];
              uint32_t addr[U];
              bool ok[U];
#pragma unroll
              for (int u = 0; u < U; ++u) {
                const int hx = slot + kXfSlots * (u0 + u);
                const int r = hy * pitch + hx;                 // 128-byte row of the stage
                ok[u] = hx >= hx_lo && hx < hx_hi;
                addr[u] = st_s + (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4));
                if (ok[u]) asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(raw[u][0]), "=r"(raw[u][1]), "=r"(raw[u][2]), "=r"(raw[u][3]) : "r"(addr[u]));
              }
#pragma unroll
              for (int u = 0; u < U; ++u) {
                if (ok[u]) {
                  uint32_t o[4];
#pragma unroll
                  for (int k = 0; k < 4; ++k) {
                    uint32_t a;
                    asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(a) : "r"(raw[u][k]), "r"(sc2[k]), "r"(sh2[k]));
                    if (swish) {
                      uint32_t h, tt;
                      asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(h) : "r"(a), "r"(0x3f003f00u));      // 0.5, 0.5
                      asm("tanh.approx.bf16x2 %0, %1;" : "=r"(tt) : "r"(h));
                      asm("fma.rn.bf16x2 %0, %1, %2, %1;" : "=r"(a) : "r"(h), "r"(tt));
                    }
                    o[k] = a;
                  }
                  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr[u]), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
                }
              }
             }
            }
            // one arrival per WARP (per-thread arrivals on one shared-memory word serialise)
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&row_rdy[sa * kRowMax + hy]);
          }
          ph_row ^= 1u << sa;
          if (++sa == kRingA) { sa = 0; pa ^= 1; }
        }
        // fused 1x1 segment (ResnetBlock res_conv): the raw x2 tile passes through untouched
        for (int ei = p.n_taps; ei < p.n_entries; ++ei) {
          const int n2 = p.e[ei].nchunks;
          for (int c = 0; c < n2; ++c) {
            mbar_wait(&full_raw[sa], (ph_x2 >> sa) & 1u);
            ph_x2 ^= 1u << sa;
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_a[sa]);
            if (++sa == kRingA) { sa = 0; pa ^= 1; }
          }
        }
      }
      (void)pa;
    }
  } else {
    // ===================== epilogue (warps 0..7) =====================
    if constexpr (FUSE) asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int row = quad * 32 + lane;          // row of the 128-row tile
    constexpr int kChunksPerWarp = BLOCK_N / 32 / (kEpiWarps / 4);
    const int ch_begin = (warp >> 2) * kChunksPerWarp;
    const int rows_box = HALO ? p.t1 : p.t1 * p.t2 * p.t3;
    // GroupNorm statistics accumulated in registers across consecutive tiles of the same (image, column tile):
    // lane j of this warp owns column n0 + j of every 32-column chunk
    float st_s[kChunksPerWarp], st_q[kChunksPerWarp];
#pragma unroll
    for (int i = 0; i < kChunksPerWarp; ++i) { st_s[i] = 0.f; st_q[i] = 0.f; }
    // STG: statistics are read back from the staged bf16 tile two columns at a time: lane l accumulates columns
    // 2*(l & 15), +1 over the rows of parity l >> 4 (st_s / st_q hold the even column, st_s1 / st_q1 the odd one)
    float st_s1[STG ? kChunksPerWarp : 1], st_q1[STG ? kChunksPerWarp : 1];
#pragma unroll
    for (int i = 0; i < (STG ? kChunksPerWarp : 1); ++i) { st_s1[i] = 0.f; st_q1[i] = 0.f; }
    // kRegStats (the warp owns ONE 32-column chunk, i.e. N = 64): only the FIRST exchange round of the transpose-reduce
    // runs per output row; its 16 partial sums per statistic are accumulated in registers and the remaining four rounds
    // run once per image.  (The full per-row reduce was ~half of all issue slots of the N = 64 kernels and left their
    // epilogue exposed; keeping all 32 columns per thread instead would need 64 more registers than the 168 available.)
    // (measured on B200: the register-accumulated variant is SLOWER than the per-row reduce -- 0.24 vs 0.21 ms epilogue-only on the
    // 64->64 layer -- because 32 more live registers push the 168-register epilogue into local-memory spills; kept for reference)
    constexpr bool kRegStats = false && kChunksPerWarp == 1;
    float rs_s[kRegStats ? 16 : 1], rs_q[kRegStats ? 16 : 1];
#pragma unroll
    for (int j = 0; j < (kRegStats ? 16 : 1); ++j) { rs_s[j] = 0.f; rs_q[j] = 0.f; }
    int st_img = -1, st_nt = -1;
    auto flush_stats = [&]() {
      if constexpr (kRegStats) {
        if (st_img >= 0) {
#pragma unroll
          for (int off = 8; off >= 1; off >>= 1) {
            const bool upper = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < off; ++i) {
              const float send_s = upper ? rs_s[i] : rs_s[i + off];
              const float keep_s = upper ? rs_s[i + off] : rs_s[i];
              const float send_q = upper ? rs_q[i] : rs_q[i + off];
              const float keep_q = upper ? rs_q[i + off] : rs_q[i];
              rs_s[i] = keep_s + __shfl_xor_sync(0xffffffffu, send_s, off);
              rs_q[i] = keep_q + __shfl_xor_sync(0xffffffffu, send_q, off);
            }
          }
          st_s[0] = rs_s[0]; st_q[0] = rs_q[0];
#pragma unroll
          for (int j = 0; j < 16; ++j) { rs_s[j] = 0.f; rs_q[j] = 0.f; }
        }
      }
      if constexpr (STG) {
        if (st_img >= 0) {
#pragma unroll
          for (int i = 0; i < kChunksPerWarp; ++i) {
            // row parities: lane l + lane l ^ 16; then lane j picks column j = component j & 1 of pair j >> 1
            const float a0 = st_s[i] + __shfl_xor_sync(0xffffffffu, st_s[i], 16), a1 = st_s1[i] + __shfl_xor_sync(0xffffffffu, st_s1[i], 16);
            const float b0 = st_q[i] + __shfl_xor_sync(0xffffffffu, st_q[i], 16), b1 = st_q1[i] + __shfl_xor_sync(0xffffffffu, st_q1[i], 16);
            const float c0 = __shfl_sync(0xffffffffu, a0, lane >> 1), c1 = __shfl_sync(0xffffffffu, a1, lane >> 1);
            const float d0 = __shfl_sync(0xffffffffu, b0, lane >> 1), d1 = __shfl_sync(0xffffffffu, b1, lane >> 1);
            st_s[i] = (lane & 1) ? c1 : c0;
            st_q[i] = (lane & 1) ? d1 : d0;
            st_s1[i] = 0.f; st_q1[i] = 0.f;
          }
        }
      }
      if (st_img >= 0 && st_img < p.M3) {
#pragma unroll
        for (int i = 0; i < kChunksPerWarp; ++i) {
          const int col = st_nt * BLOCK_N + (ch_begin + i) * 32 + lane;
          if (col < p.Ncols) {
            double* sp = p.stats + (long long)st_img * p.stats_ld + (long long)col * 2;
            atomicAdd(sp, (double)st_s[i]);
            atomicAdd(sp + 1, (double)st_q[i]);
          }
          st_s[i] = 0.f; st_q[i] = 0.f;
        }
      }
    };
    // halo mode (one image per tile): bias[c] + rowvec[image][c] of this warp's columns are staged once per tile in a
    // private slice of shared memory and re-read as broadcast vectors for every output row (with 227 KB of shared memory
    // carved out there is almost no L1 left, so the per-row __ldg's of the classic path were L2 round trips)
    float* bs = (float*)(smem + Cfg::kSmemData + 512) + warp * (32 * kChunksPerWarp);
    int it = 0;
    for (int tq = tile_begin; tq < tile_end; ++tq, ++it) {
      const int tile = work_tile(tq);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const TileCoord t = decode_tile(p, tile);
      const int nt = t.nt, i1 = t.i1, i2 = t.i2, i3 = t.i3, zb = t.zb;
      float bs_reg[HALO ? kChunksPerWarp : 1];
      if constexpr (HALO) {
#pragma unroll
        for (int ci = 0; ci < kChunksPerWarp; ++ci) {
          const int col = nt * BLOCK_N + (ch_begin + ci) * 32 + lane;
          float vb = 0.f;
          if (col < p.Ncols) {
            if (p.bias) vb += __ldg(p.bias + col);
            if (p.rowvec) vb += __ldg(p.rowvec + (long long)i3 * p.rowvec_ld + col);
          }
          bs_reg[ci] = vb;
        }
      }
      if (p.stats != nullptr) {
        const int img_w = i3 * p.t3 + (HALO ? 0 : (quad * 32) / (p.t1 * p.t2));     // warp-uniform
        if (img_w != st_img || nt != st_nt) { flush_stats(); st_img = img_w; st_nt = nt; }
      }

      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if constexpr (HALO) {
        __syncwarp();
#pragma unroll
        for (int ci = 0; ci < kChunksPerWarp; ++ci) bs[ci * 32 + lane] = bs_reg[ci];
        __syncwarp();
      }
      if constexpr (SPLIT) {
        // this CTA's MMAs are complete: its operand ring is dead.  Tell the whole cluster, then wait until every ring is (the
        // partials land in the rings).
        const uint32_t S = (uint32_t)p.ksplit;
        if (warp == 0 && (uint32_t)lane < S) mbar_arrive_remote_release(done_bar, (uint32_t)lane);
        mbar_wait_cluster(done_bar, 0);
        // phase A: the chunks another CTA finishes go to that CTA's shared memory as fp32 partials: slot (chunk / S, source), one
        // 128-byte row per lane, 16-byte pieces XOR-swizzled by the row so that a warp's stores spread over all banks
        const uint32_t ring = smem_u32(smem);
#pragma unroll 1
        for (int ci = 0; ci < kChunksPerWarp; ++ci) {
          const int ch = ch_begin + ci;
          const uint32_t owner = (uint32_t)ch % S;
          if (owner == (uint32_t)split_s) continue;
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * Cfg::kAccCols + ch * 32), v);
          const uint32_t src_idx = (uint32_t)split_s < owner ? (uint32_t)split_s : (uint32_t)split_s - 1u;
          const uint32_t slot = ((uint32_t)(ch / (int)S) * (S - 1u) + src_idx) * (uint32_t)(kBlockM * 128) + (uint32_t)row * 128u;
          const uint32_t dst = dsmem_addr(ring + slot, owner);
#pragma unroll
          for (int q = 0; q < 8; ++q) dsmem_st4(dst + (uint32_t)((q ^ (row & 7)) << 4), v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
        fence_acq_rel_cluster();
        __syncwarp();
        if ((uint32_t)lane < S && lane != split_s) mbar_arrive_remote_release(recv_bar, (uint32_t)lane);
        mbar_wait_cluster(recv_bar, 0);
      }
#pragma unroll 1
      for (int rr = 0; rr < ROWS; ++rr) {
      // row -> coordinates
      const int l1 = HALO ? row : row % p.t1;
      const int l2 = HALO ? rr : (row / p.t1) % p.t2;
      const int l3 = HALO ? 0 : row / (p.t1 * p.t2);
      const int r1 = i1 * p.t1 + l1, r2 = i2 * (HALO ? ROWS : p.t2) + l2, r3 = i3 * p.t3 + l3;
      const bool row_ok = row < rows_box && r1 < p.M1 && r2 < p.M2 && r3 < p.M3;
      const long long o1 = (long long)r1 * p.mul1 + p.off1, o2 = (long long)r2 * p.mul2 + p.off2;
      const long long obase = o1 * p.o_s1 + o2 * p.o_s2 + (long long)r3 * p.o_s3 + (long long)zb * p.o_sb;
      const long long rbase = o1 * p.r_s1 + o2 * p.r_s2 + (long long)r3 * p.r_s3 + (long long)zb * p.r_sb;
      const long long qbase = o1 * p.q_s1 + o2 * p.q_s2 + (long long)r3 * p.q_s3 + (long long)zb * p.q_sb;
      const float* rowvec = p.rowvec ? p.rowvec + (long long)r3 * p.rowvec_ld : nullptr;
#pragma unroll 1
      for (int ci = 0; ci < kChunksPerWarp; ++ci) {
        const int ch = ch_begin + ci;
        if constexpr (SPLIT) { if (ch % p.ksplit != split_s) continue; }
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * Cfg::kAccCols + rr * BLOCK_N + ch * 32), v);
        if constexpr (SPLIT) {
          // phase B: this CTA owns the chunk -- add the other CTAs' partials out of the ring
          const int S = p.ksplit;
          for (int si = 0; si < S - 1; ++si) {
            const uint8_t* src = smem + ((size_t)((ch / S) * (S - 1) + si) * kBlockM + row) * 128;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t4 = *(const float4*)(src + ((q ^ (row & 7)) << 4));
              v[4 * q] = __float_as_uint(__uint_as_float(v[4 * q]) + t4.x); v[4 * q + 1] = __float_as_uint(__uint_as_float(v[4 * q + 1]) + t4.y);
              v[4 * q + 2] = __float_as_uint(__uint_as_float(v[4 * q + 2]) + t4.z); v[4 * q + 3] = __float_as_uint(__uint_as_float(v[4 * q + 3]) + t4.w);
            }
          }
        }
        const int n0 = nt * BLOCK_N + ch * 32;
        if constexpr (STG) {
          // ---- staged epilogue: 32 full bf16 columns; residual loads and output stores go through the warp's staging buffer
          // with four lanes per row (8 lines per instruction instead of 32) ----
          uint8_t* stg = smem + Cfg::kSmemData + 512 + Cfg::kBsumBytes + warp * 1024;
          const int my16 = lane & 15;                                   // my row inside a 16-row half
          const int mysw = (my16 >> 1) & 3;
          const int sr = lane >> 2, sq = lane & 3;                      // store layout: 8 rows x four 16-byte columns per pass
          // the residual does not depend on the accumulator: fetch it first so that its latency hides behind the TMEM load
          uint4 rv[4];
          if (p.res) {
#pragma unroll
            for (int hj = 0; hj < 4; ++hj) {
              const int src = 8 * hj + sr;
              long long rb; int ok;
              if constexpr (HALO) {       // a warp's rows are consecutive pixels of one image row: addresses are linear in the row index
                rb = rbase + (long long)(src - lane) * p.mul1 * p.r_s1;
                ok = (quad * 32 + src < rows_box) && (i1 * p.t1 + quad * 32 + src < p.M1) && r2 < p.M2 && r3 < p.M3;
              } else {
                rb = __shfl_sync(0xffffffffu, rbase, src);
                ok = __shfl_sync(0xffffffffu, (int)row_ok, src);
              }
              rv[hj] = make_uint4(0u, 0u, 0u, 0u);
              if (ok) rv[hj] = __ldg((const uint4*)((const __nv_bfloat16*)p.res + rb + n0 + sq * 8));
            }
          }
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          if constexpr (HALO) {
            const float4* b4 = (const float4*)(bs + ci * 32);
#pragma unroll
            for (int q = 0; q < 8; ++q) { float4 t4 = b4[q]; f[4 * q] += t4.x; f[4 * q + 1] += t4.y; f[4 * q + 2] += t4.z; f[4 * q + 3] += t4.w; }
          } else {
            if (p.bias) {
              const float4* b4 = (const float4*)(p.bias + n0);
#pragma unroll
              for (int q = 0; q < 8; ++q) { float4 t4 = __ldg(b4 + q); f[4 * q] += t4.x; f[4 * q + 1] += t4.y; f[4 * q + 2] += t4.z; f[4 * q + 3] += t4.w; }
            }
            if (rowvec && row_ok) {
              const float4* r4 = (const float4*)(rowvec + n0);
#pragma unroll
              for (int q = 0; q < 8; ++q) { float4 t4 = __ldg(r4 + q); f[4 * q] += t4.x; f[4 * q + 1] += t4.y; f[4 * q + 2] += t4.z; f[4 * q + 3] += t4.w; }
            }
          }
          if (p.act != WSR_ACT_NONE) {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = apply_act(f[j], p.act);
          }
          if (p.out_scale != 1.f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] *= p.out_scale;
          }
          if (p.res) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const int r16 = 8 * j + sr;
                *(uint4*)(stg + r16 * 64 + ((sq ^ ((r16 >> 1) & 3)) << 4)) = rv[2 * h + j];
              }
              __syncwarp();
              if ((lane >> 4) == h) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const uint4 u = *(const uint4*)(stg + my16 * 64 + ((q ^ mysw) << 4));
                  const __nv_bfloat162* hh = (const __nv_bfloat162*)&u;
#pragma unroll
                  for (int k = 0; k < 4; ++k) { float2 t2 = __bfloat1622float2(hh[k]); f[q * 8 + 2 * k] += p.res_scale * t2.x; f[q * 8 + 2 * k + 1] += p.res_scale * t2.y; }
                }
              }
              __syncwarp();
            }
          }
          uint4 pk[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            __nv_bfloat162* hh = (__nv_bfloat162*)&pk[q];
#pragma unroll
            for (int k = 0; k < 4; ++k) hh[k] = row_ok ? __floats2bfloat162_rn(f[q * 8 + 2 * k], f[q * 8 + 2 * k + 1]) : __floats2bfloat162_rn(0.f, 0.f);
          }
          float cs0 = 0.f, cs1 = 0.f, cq0 = 0.f, cq1 = 0.f;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if ((lane >> 4) == h) {
#pragma unroll
              for (int q = 0; q < 4; ++q) *(uint4*)(stg + my16 * 64 + ((q ^ mysw) << 4)) = pk[q];
            }
            __syncwarp();
            if (p.stats != nullptr) {
              // lane l: columns 2*(l & 15), +1 of the rows with parity l >> 4 (rows r and r + 1 sit in different 64-byte halves
              // of the 128-byte bank window: conflict-free)
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int r = 2 * i + (lane >> 4);
                const __nv_bfloat162 x2 = *(const __nv_bfloat162*)(stg + r * 64 + ((((lane & 15) >> 2) ^ ((r >> 1) & 3)) << 4) + (lane & 3) * 4);
                const float2 x = __bfloat1622float2(x2);
                cs0 += x.x; cq0 = fmaf(x.x, x.x, cq0);
                cs1 += x.y; cq1 = fmaf(x.y, x.y, cq1);
              }
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const int src = 16 * h + 8 * j + sr;
              long long ob; int ok;
              if constexpr (HALO) {
                ob = obase + (long long)(src - lane) * p.mul1 * p.o_s1;
                ok = (quad * 32 + src < rows_box) && (i1 * p.t1 + quad * 32 + src < p.M1) && r2 < p.M2 && r3 < p.M3;
              } else {
                ob = __shfl_sync(0xffffffffu, obase, src);
                ok = __shfl_sync(0xffffffffu, (int)row_ok, src);
              }
              const int r16 = 8 * j + sr;
              const uint4 u = *(const uint4*)(stg + r16 * 64 + ((sq ^ ((r16 >> 1) & 3)) << 4));
              if (ok) *(uint4*)((__nv_bfloat16*)p.out + ob + n0 + sq * 8) = u;
            }
            __syncwarp();
          }
          if (p.stats != nullptr) {
#pragma unroll
            for (int i = 0; i < kChunksPerWarp; ++i)
              if (i == ci) { st_s[i] += cs0; st_q[i] += cq0; st_s1[i] += cs1; st_q1[i] += cq1; }
          }
        } else {
          float f[32];
  #pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = 0.f;
          if (row_ok && n0 < p.Ncols) {
            const bool full = (n0 + 32 <= p.Ncols);
  #pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
            if constexpr (HALO) {
              const float4* b4 = (const float4*)(bs + ci * 32);
  #pragma unroll
              for (int q = 0; q < 8; ++q) { float4 t4 = b4[q]; f[4 * q] += t4.x; f[4 * q + 1] += t4.y; f[4 * q + 2] += t4.z; f[4 * q + 3] += t4.w; }
            } else if (full) {
              // 32 consecutive columns: bias / time-embedding row as independent 16-byte loads (same address in every
              // lane -> one broadcast transaction each), issued back to back
              if (p.bias) {
                const float4* b4 = (const float4*)(p.bias + n0);
  #pragma unroll
                for (int q = 0; q < 8; ++q) { float4 t4 = __ldg(b4 + q); f[4 * q] += t4.x; f[4 * q + 1] += t4.y; f[4 * q + 2] += t4.z; f[4 * q + 3] += t4.w; }
              }
              if (rowvec) {
                const float4* r4 = (const float4*)(rowvec + n0);
  #pragma unroll
                for (int q = 0; q < 8; ++q) { float4 t4 = __ldg(r4 + q); f[4 * q] += t4.x; f[4 * q + 1] += t4.y; f[4 * q + 2] += t4.z; f[4 * q + 3] += t4.w; }
              }
            } else {
  #pragma unroll
              for (int j = 0; j < 32; ++j)
                if (n0 + j < p.Ncols) {
                  if (p.bias) f[j] += __ldg(p.bias + n0 + j);
                  if (rowvec) f[j] += __ldg(rowvec + n0 + j);
                }
            }
            if (p.act != WSR_ACT_NONE) {
  #pragma unroll
              for (int j = 0; j < 32; ++j) f[j] = apply_act(f[j], p.act);
            }
            if (p.out_scale != 1.f) {
  #pragma unroll
              for (int j = 0; j < 32; ++j) f[j] *= p.out_scale;
            }
            const bool vec_ok = full && p.o_sc == 1 && ((obase + n0) & 7) == 0 && (((uintptr_t)p.out) & 15) == 0;
            if (p.res) {
              if (full && p.r_sc == 1 && p.res_dtype == WSR_BF16 && ((rbase + n0) & 7) == 0 && (((uintptr_t)p.res) & 15) == 0) {
                const uint4* rp = (const uint4*)((const __nv_bfloat16*)p.res + rbase + n0);
  #pragma unroll
                for (int q = 0; q < 4; ++q) {
                  uint4 u = rp[q];
                  const __nv_bfloat162* h = (const __nv_bfloat162*)&u;
  #pragma unroll
                  for (int k = 0; k < 4; ++k) { float2 t2 = __bfloat1622float2(h[k]); f[q * 8 + 2 * k] += p.res_scale * t2.x; f[q * 8 + 2 * k + 1] += p.res_scale * t2.y; }
                }
              } else {
  #pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (n0 + j < p.Ncols) f[j] += p.res_scale * ld_dt(p.res, rbase + (long long)(n0 + j) * p.r_sc, p.res_dtype);
              }
            }
            if (p.res2) {
  #pragma unroll
              for (int j = 0; j < 32; ++j)
                if (n0 + j < p.Ncols) f[j] += p.res2_scale * ld_dt(p.res2, qbase + (long long)(n0 + j) * p.q_sc, p.res2_dtype);
            }
            if (vec_ok && p.out_dtype == WSR_BF16) {
              uint4* op = (uint4*)((__nv_bfloat16*)p.out + obase + n0);
  #pragma unroll
              for (int q = 0; q < 4; ++q) {
                uint4 u;
                __nv_bfloat162* h = (__nv_bfloat162*)&u;
  #pragma unroll
                for (int k = 0; k < 4; ++k) h[k] = __floats2bfloat162_rn(f[q * 8 + 2 * k], f[q * 8 + 2 * k + 1]);
                op[q] = u;
              }
            } else if (vec_ok && p.out_dtype == WSR_F32) {
              float4* op = (float4*)((float*)p.out + obase + n0);
  #pragma unroll
              for (int q = 0; q < 8; ++q) op[q] = make_float4(f[4 * q], f[4 * q + 1], f[4 * q + 2], f[4 * q + 3]);
            } else {
  #pragma unroll
              for (int j = 0; j < 32; ++j)
                if (n0 + j < p.Ncols) st_dt(p.out, obase + (long long)(n0 + j) * p.o_sc, p.out_dtype, f[j]);
            }
          }
          __syncwarp();
          if constexpr (kRegStats) {
            if (p.stats != nullptr && n0 < p.Ncols) {
              // first round (offset 16): lanes with bit 4 clear keep columns 0..15, the others 16..31
              const bool upper = (lane & 16) != 0;
  #pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float lo = f[i], hi = f[i + 16];
                const float send_s = upper ? lo : hi, keep_s = upper ? hi : lo;
                const float got_s = __shfl_xor_sync(0xffffffffu, send_s, 16);
                const float got_q = __shfl_xor_sync(0xffffffffu, send_s * send_s, 16);
                rs_s[i] += keep_s + got_s;
                rs_q[i] += fmaf(keep_s, keep_s, got_q);
              }
            }
          } else
          if (p.stats != nullptr && n0 < p.Ncols) {
            // per-channel sum / sum of squares over the warp's 32 rows: transpose-reduce with 31 shuffles per statistic so
            // that lane j ends up with column n0 + j; masked rows hold zeros
            float q2[32];
  #pragma unroll
            for (int j = 0; j < 32; ++j) q2[j] = f[j] * f[j];
  #pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
              const bool upper = (lane & off) != 0;
  #pragma unroll
              for (int i = 0; i < off; ++i) {
                const float send_s = upper ? f[i] : f[i + off];
                const float keep_s = upper ? f[i + off] : f[i];
                const float send_q = upper ? q2[i] : q2[i + off];
                const float keep_q = upper ? q2[i + off] : q2[i];
                f[i] = keep_s + __shfl_xor_sync(0xffffffffu, send_s, off);
                q2[i] = keep_q + __shfl_xor_sync(0xffffffffu, send_q, off);
              }
            }
  #pragma unroll
            for (int i = 0; i < kChunksPerWarp; ++i)
              if (i == ci) { st_s[i] += f[0]; st_q[i] += q2[0]; }
          }
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if constexpr (PAIR) mbar_arrive_leader(&tempty_bar[acc]); else mbar_arrive(&tempty_bar[acc]); }
    }
    if (p.stats != nullptr) flush_stats();
  }

  tc_fence_before();
  // PAIR: neither CTA may leave (or free tensor memory) while the other can still signal its barriers or its MMAs read its B half
  if constexpr (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::kTmemCols) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

// bf16 tensor map, rank `rank`, innermost box 64 elements (128 B) with 128B swizzle
int encode_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  WSR_REQUIRE(enc != nullptr, WSR_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i < rank - 1; ++i) gs[i] = strides_bytes[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  WSR_REQUIRE(r == CUDA_SUCCESS, WSR_E_CUDA,
              "cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu %llu %llu %llu] strides [%llu %llu %llu] box [%u %u %u %u] base %p",
              (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)(rank > 2 ? dims[2] : 0),
              (unsigned long long)(rank > 3 ? dims[3] : 0), (unsigned long long)strides_bytes[0],
              (unsigned long long)(rank > 2 ? strides_bytes[1] : 0), (unsigned long long)(rank > 3 ? strides_bytes[2] : 0), box[0],
              box[1], rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0, base);
  return WSR_OK;
}

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int BLOCK_N, bool HALO, int ROWS, bool FUSE = false, bool VM = false, bool STG = false, bool SPLIT = false>
static int launch_tc_impl(const TcParams& p, cudaStream_t st) {
  using Cfg = TcCfg<BLOCK_N, HALO, ROWS, VM>;
  static bool attr_set = false;
  if (!attr_set) {
    WSR_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<BLOCK_N, HALO, ROWS, FUSE, VM, STG, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  const int total = p.g1 * p.g2 * p.g3 * p.nbatch * p.n_tiles;
  if constexpr (SPLIT) {
    // one cluster of ksplit CTAs per tile (CTA rank in the cluster = K range)
    WSR_REQUIRE(p.ksplit >= 2 && p.ksplit <= 8 && p.ksplit <= BLOCK_N / 32 && (BLOCK_N / 32) % p.ksplit == 0, WSR_E_INVALID, "gemm_tc: split-K launch invariants");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(total * p.ksplit);
    cfg.blockDim = dim3(kTcThreads);
    cfg.dynamicSmemBytes = (size_t)Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)p.ksplit; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    WSR_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BLOCK_N, HALO, ROWS, FUSE, VM, STG, SPLIT>, p));
  } else {
    const int grid = total < sm_count() ? total : sm_count();
    WSR_CUDA_OK(launch_pdl(gemm_tc_kernel<BLOCK_N, HALO, ROWS, FUSE, VM, STG, SPLIT>, dim3(grid), dim3(FUSE ? kTcThreadsFused : kTcThreads),
                           (size_t)Cfg::kSmemBytes, st, p));
  }
  return WSR_OK;
}

// CTA-pair launch: a row of 2-CTA clusters, at most one pair per TPC the device can co-schedule (asked from the occupancy API once)
template <bool STG>
static int launch_tc_pair(const TcParams& p, cudaStream_t st) {
  using Cfg = TcCfg<256, false, 1, false, true>;
  auto kern = gemm_tc_kernel<256, false, 1, false, false, STG, false, true>;
  static int max_pairs = 0;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = (size_t)Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  if (!max_pairs) {
    WSR_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    cfg.gridDim = dim3(sm_count() / 2 * 2);
    cfg.numAttrs = 1;
    int n = 0;
    WSR_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    WSR_REQUIRE(n > 0, WSR_E_CUDA, "gemm_tc: the device cannot co-schedule a CTA pair of the 256-column kernel");
    max_pairs = n < sm_count() / 2 ? n : sm_count() / 2;
  }
  const int total = p.g1 * p.g2 * p.g3 * p.nbatch * p.n_tiles;
  WSR_REQUIRE(total % 2 == 0 && (p.g1 * p.g2 * p.g3 * p.nbatch) % 2 == 0, WSR_E_INVALID, "gemm_tc: CTA pairs need an even number of row tiles");
  const int pairs = total / 2 < max_pairs ? total / 2 : max_pairs;
  cfg.gridDim = dim3(2 * pairs);
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  WSR_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, p));
  return WSR_OK;
}

// Preconditions of the staged epilogue (STG kernels): bf16 output (and residual) with unit channel stride, every row start
// 16-byte aligned, whole 32-column chunks only.
static bool stage_preconditions(const TcParams& p, int block_n) {
  auto m8 = [](long long v) { return (v & 7) == 0; };
  if (p.out_dtype != WSR_BF16 || p.o_sc != 1 || (((uintptr_t)p.out) & 15) != 0 || p.Ncols % block_n != 0 || p.res2 != nullptr) return false;
  if (!(m8(p.o_s1) && m8(p.o_s2) && m8(p.o_s3) && m8(p.o_sb))) return false;
  if (p.res) {
    if (p.res_dtype != WSR_BF16 || p.r_sc != 1 || (((uintptr_t)p.res) & 15) != 0) return false;
    if (!(m8(p.r_s1) && m8(p.r_s2) && m8(p.r_s3) && m8(p.r_sb))) return false;
  }
  return true;
}

template <int BLOCK_N>
static int launch_tc(const TcParams& p, cudaStream_t st) {
  const bool sok = stage_preconditions(p, BLOCK_N);
  if (p.n_taps > 0 && p.gn_tab != nullptr) {
    // fused GroupNorm input: the same tile shapes as the plain halo kernels (vertical tap merge for N = 64, two rows for N = 128),
    // staged epilogue whenever its preconditions hold
    if constexpr (BLOCK_N == 64) {
      if (p.halo_rows == 3) return sok ? launch_tc_impl<BLOCK_N, true, 3, true, true, true>(p, st) : launch_tc_impl<BLOCK_N, true, 3, true, true>(p, st);
    }
    if constexpr (BLOCK_N <= 128) {
      if (p.halo_rows == 2) return sok ? launch_tc_impl<BLOCK_N, true, 2, true, false, true>(p, st) : launch_tc_impl<BLOCK_N, true, 2, true>(p, st);
    }
    WSR_REQUIRE(p.halo_rows == 1, WSR_E_INVALID, "conv_tc: fused GroupNorm input with %d halo rows", p.halo_rows);
    return sok ? launch_tc_impl<BLOCK_N, true, 1, true, false, true>(p, st) : launch_tc_impl<BLOCK_N, true, 1, true>(p, st);
  }
  if (p.n_taps > 0) {
    if constexpr (BLOCK_N == 64) {
      if (p.halo_rows == 3) return sok ? launch_tc_impl<BLOCK_N, true, 3, false, true, true>(p, st) : launch_tc_impl<BLOCK_N, true, 3, false, true>(p, st);
    }
    if constexpr (BLOCK_N <= 64) {
      if (p.halo_rows == 4) return launch_tc_impl<BLOCK_N, true, 4>(p, st);
    }
    if constexpr (BLOCK_N <= 128) {
      if (p.halo_rows == 2) return sok ? launch_tc_impl<BLOCK_N, true, 2, false, false, true>(p, st) : launch_tc_impl<BLOCK_N, true, 2>(p, st);
    }
    return sok ? launch_tc_impl<BLOCK_N, true, 1, false, false, true>(p, st) : launch_tc_impl<BLOCK_N, true, 1>(p, st);
  }
  if (p.ksplit > 1) {
    // pick_split only cuts launches whose tiles fit in half a wave, and pick_block_n gives those 64-column tiles
    WSR_REQUIRE(BLOCK_N == 64 && p.ksplit == 2 && sok, WSR_E_INVALID, "gemm_tc: split-K chosen with BN=%d S=%d or without the staged-epilogue preconditions",
                BLOCK_N, p.ksplit);
    if constexpr (BLOCK_N == 64) return launch_tc_impl<BLOCK_N, false, 1, false, false, true, true>(p, st);
  }
  if constexpr (BLOCK_N == 256) {
    if (p.pair) return sok ? launch_tc_pair<true>(p, st) : launch_tc_pair<false>(p, st);
  }
  if (sok) return launch_tc_impl<BLOCK_N, false, 1, false, false, true>(p, st);
  return launch_tc_impl<BLOCK_N, false, 1>(p, st);
}

// Split-K for a classic-mode launch whose tiles do not fill the machine (deep UNet levels at small batch: 8 .. 64 row tiles for 148 SMs).
// What bounds such a launch is the operand fetch of each CTA -- one SM receives at most ~65 bytes per clock from L2 (tools/tma_probe.cu,
// profiles/r02_tma_probe.txt) -- or its MMAs; cutting the K loop over the CTAs of a cluster divides both, at the price of the
// partial-tile exchange through distributed shared memory.
// MEASURED on B200 (tools/prof_conv.py, profiles/r02_splitk_cluster_sweep.txt; 512->512 3x3 @8x16, 8 images, unsplit BN = 64: 24.7 us):
// BN 64 / S 2: 21.1 us, BN 128 / S 2 and S 4: 22.9 / 22.7 us, BN 256 / S 2 and S 4: 27.3 us, BN 256 / S 8: 56 us.  The launch is
// t = 5.3 us + 0.27 us per K block; halving the K loop saves 9.7 us and the cluster launch + two cluster-wide barrier rounds + the
// exchange give 6 us of it back, and clusters of 8 do not even fit one wave.  Whole step at 8 images per GPU: 3.38 ms without, 3.90 ms
// with a cost-model search over (BN, S) and S up to 8.  So the rule is the single cut that measured faster: keep the unsplit tile shape and
// halve its K loop over a 2-CTA cluster, when that still fits one wave and the K loop is long enough to pay for the exchange (3x3
// convolutions with >= 256 input channels: 24.7 -> 21.1 us, 43.7 -> 33.8 us, 28.8 -> 24.0 us on the 8x16 level at 8 images; 1x1
// convolutions get SLOWER, 7.5 -> 9.6 us).  (The round-1 global-memory exchange was worse still: 30 us.)
// Tiles that fit in half a wave always get BN = 64 from pick_block_n, so a split launch has BN = 64 and S = 2.  Returns S (1 = no split).
static int pick_split(int ncols, int m_tiles, int total_kb, int bn) {
  const int tiles = m_tiles * ((ncols + bn - 1) / bn);
  return (total_kb >= 36 && 2 * tiles <= sm_count() && ncols % bn == 0) ? 2 : 1;
}

static int g_last_ksplit = 1, g_last_bn = 0, g_last_pair = 0;      // introspection for the tests (wsr_debug_last_tc_config)
static int g_pair_mode = 1;                       // CTA-pair policy, see wsr_debug_set_pair

static int pick_block_n(int ncols, int m_tiles) {
  // Column-tile width by a small cost model measured on B200: one 128 x BN x 16 MMA costs about (69 + 0.28 * BN) cycles
  // (the 128-row activation operand fetch is the fixed part), and a launch needs ceil(tiles / SMs) waves.  E.g. the 8x16
  // level at B = 64 (64 row tiles, Cout = 512): BN = 256 -> 128 tiles = ONE 86%-full wave of 141-cycle MMAs beats
  // BN = 128 -> 256 tiles = two waves of 105-cycle MMAs.
  const int sms = sm_count();
  const int cand[3] = {256, 128, 64};
  int best = 64;
  double best_cost = 1e30;
  for (int i = 0; i < 3; ++i) {
    const int bn = cand[i];
    if (ncols % bn != 0 && !(bn == 64)) continue;
    const int tiles = m_tiles * ((ncols + bn - 1) / bn);
    const int waves = (tiles + sms - 1) / sms;
    const double cost = (double)waves * (69.0 + 0.28 * bn);
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

int validate_conv_desc(const WsrConvDesc* d);
int validate_gemm_desc(const WsrGemmDesc* g);
int validate_taps(const WsrTapTable* t);

static void choose_tile(int W, int H, int N, int& t1, int& t2, int& t3) {
  t1 = W < 128 ? W : 128;
  t2 = 128 / t1; if (t2 > H) t2 = H; if (t2 < 1) t2 = 1;
  t3 = 128 / (t1 * t2); if (t3 > N) t3 = N; if (t3 < 1) t3 = 1;
}

}  // namespace wsr

using namespace wsr;

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

/* (column-tile width << 8) | K splits of the most recent wsr_conv_tc / wsr_conv_taps_tc launch of this process (tests only) */
extern "C" int wsr_debug_last_tc_config(void) { return (g_last_pair << 20) | (g_last_bn << 8) | g_last_ksplit; }
// CTA-pair policy of the classic 256-column convolution tiles: 0 never, 1 launches of more than one wave (default), 2 every eligible launch
extern "C" int wsr_debug_set_pair(int mode) {
  const int prev = g_pair_mode; g_pair_mode = mode < 0 ? 0 : (mode > 2 ? 2 : mode); return prev;
}

extern "C" int wsr_conv_tc(const WsrConvDesc* d, void* stream) {
  int rc = validate_conv_desc(d);
  if (rc) return rc;
  WSR_REQUIRE(d->x_dtype == WSR_BF16, WSR_E_UNSUPPORTED, "conv_tc: bf16 operands only");
  WSR_REQUIRE(d->Cin % 64 == 0 && d->x_ld % 8 == 0 && (((uintptr_t)d->x) & 15) == 0 && (((uintptr_t)d->w) & 15) == 0,
              WSR_E_UNSUPPORTED, "conv_tc: Cin %% 64, pitch %% 8 and 16-byte alignment required (Cin=%d ld=%d)", d->Cin, d->x_ld);
  if (d->x2)
    WSR_REQUIRE(d->Cin2 % 64 == 0 && d->x2_ld % 8 == 0 && (((uintptr_t)d->x2) & 15) == 0 && (((uintptr_t)d->w2) & 15) == 0,
                WSR_E_UNSUPPORTED, "conv_tc: second segment Cin2 %% 64 / alignment");
  WSR_REQUIRE(!(d->x2 && (d->stride != 1 || d->upsample)), WSR_E_UNSUPPORTED, "conv_tc: second segment needs stride 1, no upsample");
  WSR_REQUIRE((((uintptr_t)d->bias) & 15) == 0 && (((uintptr_t)d->rowvec) & 15) == 0 && (d->rowvec == nullptr || d->rowvec_ld % 4 == 0),
              WSR_E_UNSUPPORTED, "conv_tc: bias / rowvec must be 16-byte aligned, rowvec_ld %% 4 == 0");
  cudaStream_t st = (cudaStream_t)stream;

  const int up = d->upsample ? 2 : 1;
  const int OH = d->H * up / d->stride, OW = d->W * up / d->stride;
  // grid of GEMM rows: output pixels (stride 1 / 2) or input-resolution pixels per output phase (upsample)
  const int GH = d->upsample ? d->H : OH, GW = d->upsample ? d->W : OW;
  const bool merged = d->upsample == 2;          // phase-merged 2x2 taps (wsr_pack_upsample_weight)
  WSR_REQUIRE(!merged || d->ksize == 3, WSR_E_UNSUPPORTED, "conv_tc: merged upsample needs ksize 3");
  const int taps = merged ? 4 : d->ksize * d->ksize;
  const int wtaps = merged ? 16 : taps;          // taps stored in the weight tensor
  const int pad = (d->ksize - 1) / 2;
  const int nphase = d->upsample ? 4 : 1;

  TcParams p;
  memset(&p, 0, sizeof(p));
  choose_tile(GW, GH, d->N, p.t1, p.t2, p.t3);
  WSR_REQUIRE(p.t1 <= 256 && p.t2 <= 256 && p.t3 <= 256, WSR_E_UNSUPPORTED, "conv_tc: tile");
  p.g1 = cdiv(GW, p.t1); p.g2 = cdiv(GH, p.t2); p.g3 = cdiv(d->N, p.t3);
  p.nbatch = 1; p.a_zmul = 0; p.b_zmul = 0;
  p.a_bytes = p.t1 * p.t2 * p.t3 * 128;
  p.M1 = GW; p.M2 = GH; p.M3 = d->N;
  p.Ncols = d->Cout;
  p.out = d->y; p.out_dtype = d->y_dtype;
  p.o_s1 = d->y_ld; p.o_s2 = (long long)OW * d->y_ld; p.o_s3 = (long long)OH * OW * d->y_ld; p.o_sb = 0; p.o_sc = 1;
  p.bias = d->bias; p.rowvec = d->rowvec; p.rowvec_ld = d->rowvec_ld;
  p.act = d->act; p.out_scale = d->out_scale;
  p.res = d->res; p.res_dtype = d->res_dtype; p.res_scale = d->res_scale;
  p.r_s1 = d->res_ld; p.r_s2 = (long long)OW * d->res_ld; p.r_s3 = (long long)OH * OW * d->res_ld; p.r_sc = 1;
  p.res2 = d->res2; p.res2_dtype = d->res2_dtype; p.res2_scale = d->res2_scale;
  p.q_s1 = d->res2_ld; p.q_s2 = (long long)OW * d->res2_ld; p.q_s3 = (long long)OH * OW * d->res2_ld; p.q_sc = 1;

  const int m_tiles = p.g1 * p.g2 * p.g3;
  const int bn = pick_block_n(d->Cout, m_tiles);
  // halo mode: when a tile is a segment of ONE image row, the 9 taps are 9 shifted views of a single halo tile, so the
  // activation operand is fetched once per 64-channel chunk instead of once per tap; with two output rows per tile
  // (two accumulators) every weight tile is used twice as well.  Both cut the L2 -> SM traffic that bounds these layers.
  const bool halo = d->ksize == 3 && d->stride == 1 && p.t2 == 1 && p.t3 == 1 && p.t1 + 2 <= 130;
  // split-K (classic tiles that do not fill the machine; needs the staged-epilogue preconditions)
  p.ksplit = 1;
  if (!halo && d->gn_table == nullptr && stage_preconditions(p, bn)) {
    const int kb_est = (merged ? 4 : taps) * (d->Cin / 64) + (d->x2 ? d->Cin2 / 64 : 0);
    p.ksplit = pick_split(d->Cout, m_tiles, kb_est, bn);
    p.kb_split = cdiv(kb_est, p.ksplit);
  }
  // vertical tap merge (N = 64, plain 3x3): three output rows per tile, needs the vmerge weight pack (w_vmerge)
  const bool vmerge = halo && bn == 64 && taps == 9 && !d->upsample && d->w_vmerge != nullptr;
  // (the 4-row tiles have no shared memory left for the staged epilogue and are not built with the fused GroupNorm input)
  const int hrows = vmerge ? 3 : (halo && bn <= 64 && GH % 4 == 0 && d->gn_table == nullptr) ? 4 : (halo && bn <= 128 && GH % 2 == 0) ? 2 : 1;
  WSR_REQUIRE(d->gn_table == nullptr || halo, WSR_E_UNSUPPORTED,
              "conv_tc: the fused GroupNorm input needs a stride-1 3x3 convolution on rows of >= 128 pixels (see wsr_conv_tc_can_fuse_gn)");
  if (d->gn_table) {
    WSR_REQUIRE(d->gn_table_ld >= d->Cin && d->gn_table_ld % 2 == 0 && (((uintptr_t)d->gn_table) & 15) == 0, WSR_E_INVALID, "conv_tc: gn_table pitch / alignment");
    WSR_REQUIRE(d->gn_act == WSR_ACT_NONE || d->gn_act == WSR_ACT_SWISH, WSR_E_UNSUPPORTED, "conv_tc: gn_act must be NONE or SWISH");
    p.gn_tab = (const float2*)d->gn_table; p.gn_ld = d->gn_table_ld; p.gn_act = d->gn_act;
    p.xg = d->x; p.xg_ld = d->x_ld; p.xg_H = d->H; p.xg_W = d->W;
    p.x2g = d->x2; p.x2g_ld = d->x2_ld;
  }
  p.n_taps = halo ? taps : 0;
  p.halo_rows = hrows;
  p.halo_bytes = (p.t1 + 2) * (hrows + 2) * 128;
  if (halo) { p.g2 = cdiv(GH, hrows); p.a_bytes = p.t1 * hrows * 128; }
  const bool fuse_stats = d->gn_stats != nullptr && (halo ? p.t1 % 32 == 0 : (p.t1 * p.t2) % 32 == 0);
  p.stats = fuse_stats ? d->gn_stats : nullptr;
  p.stats_ld = d->gn_stats_ld;

  // CTA pairs (cta_group::2) for the classic 256-column tiles: needs an even number of row tiles; wsr_debug_set_pair(2) takes every
  // eligible launch (tests)
  const int pair_mode = g_pair_mode;
  const bool pair_on = pair_mode != 0;
  // (measured on B200, tools/prof_conv.py: +6..7 % on the launches of more than one wave -- 1348 -> 1437, 1416 -> 1496, 1454 -> 1552 TFLOP/s
  // at B = 64 -- and 3..7 % SLOWER on launches of at most one wave, where neither L2 traffic nor power is the limit and the cluster launch
  // and the two cluster barriers are pure overhead: pairs only above one wave)
  p.pair = (pair_on && !halo && bn == 256 && p.ksplit == 1 && m_tiles % 2 == 0 && (pair_mode >= 2 || m_tiles * cdiv(d->Cout, bn) > sm_count())) ? 1 : 0;
  g_last_pair = p.pair;
  // ---- B maps: weights [tap][Cout][Cin]
  {
    const int wrows = d->w_rows > 0 ? d->w_rows : d->Cout;
    uint64_t dims[3] = {(uint64_t)d->Cin, (uint64_t)wrows, (uint64_t)wtaps};
    uint64_t str[2] = {(uint64_t)d->Cin * 2, (uint64_t)d->Cin * wrows * 2};
    uint32_t box[3] = {64, (uint32_t)(p.pair ? bn / 2 : bn), 1};
    rc = encode_map(&p.bmap[0], d->w, 3, dims, str, box);
    if (rc) return rc;
    p.bmap[1] = p.bmap[0];
    p.bmap[2] = p.bmap[0];
    if (vmerge) {
      // [kx][3 * 64 rows: ky = 2, 1, 0][Cin]
      uint64_t dimsv[3] = {(uint64_t)d->Cin, 192, 3};
      uint64_t strv[2] = {(uint64_t)d->Cin * 2, (uint64_t)d->Cin * 192 * 2};
      uint32_t boxv[3] = {64, 192, 1};
      WSR_REQUIRE((((uintptr_t)d->w_vmerge) & 15) == 0, WSR_E_UNSUPPORTED, "conv_tc: w_vmerge alignment");
      rc = encode_map(&p.bmap[2], d->w_vmerge, 3, dimsv, strv, boxv);
      if (rc) return rc;
    }
    if (d->x2) {
      uint64_t dims2[3] = {(uint64_t)d->Cin2, (uint64_t)wrows, 1};
      uint64_t str2[2] = {(uint64_t)d->Cin2 * 2, (uint64_t)d->Cin2 * wrows * 2};
      rc = encode_map(&p.bmap[1], d->w2, 3, dims2, str2, box);
      if (rc) return rc;
    }
  }
  // ---- A maps
  const uint32_t abox[4] = {64, (uint32_t)p.t1, (uint32_t)(halo ? hrows : p.t2), (uint32_t)p.t3};
  const long long ld = d->x_ld;
  if (d->stride == 1) {
    uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)d->W, (uint64_t)d->H, (uint64_t)d->N};
    uint64_t str[3] = {(uint64_t)ld * 2, (uint64_t)d->W * ld * 2, (uint64_t)d->H * d->W * ld * 2};
    const uint32_t hbox[4] = {64, (uint32_t)(p.t1 + 2), (uint32_t)(hrows + 2), 1};
    rc = encode_map(&p.amap[0], d->x, 4, dims, str, halo ? hbox : abox);
    if (rc) return rc;
    for (int i = 1; i < kNumAMaps; ++i) p.amap[i] = p.amap[0];
    if (halo && d->gn_table) {
      // fused GroupNorm input: the halo tile is fetched one row per TMA box (row-by-row hand-over to the transform warps)
      const uint32_t rbox[4] = {64, (uint32_t)(p.t1 + 2), 1, 1};
      rc = encode_map(&p.amap[1], d->x, 4, dims, str, rbox);
      if (rc) return rc;
    }
  } else {
    // four phase-subsampled views: phase (py, px) starts at pixel (py, px), steps 2 pixels
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)d->W / 2, (uint64_t)d->H / 2, (uint64_t)d->N};
        uint64_t str[3] = {(uint64_t)ld * 4, (uint64_t)d->W * ld * 4, (uint64_t)d->H * d->W * ld * 2};
        const __nv_bfloat16* base = (const __nv_bfloat16*)d->x + ((long long)py * d->W + px) * ld;
        rc = encode_map(&p.amap[py * 2 + px], base, 4, dims, str, abox);
        if (rc) return rc;
      }
    p.amap[4] = p.amap[0];
  }
  if (d->x2) {
    uint64_t dims[4] = {(uint64_t)d->Cin2, (uint64_t)OW, (uint64_t)OH, (uint64_t)d->N};
    uint64_t str[3] = {(uint64_t)d->x2_ld * 2, (uint64_t)OW * d->x2_ld * 2, (uint64_t)OH * OW * d->x2_ld * 2};
    rc = encode_map(&p.amap[4], d->x2, 4, dims, str, abox);
    if (rc) return rc;
  }

  for (int ph = 0; ph < nphase; ++ph) {
    const int py = ph >> 1, px = ph & 1;
    int ne = 0, kb = 0;
    const int kdim = merged ? 2 : d->ksize;
    for (int ky = 0; ky < kdim; ++ky)
      for (int kx = 0; kx < kdim; ++kx) {
        TcEntry& e = p.e[ne++];
        e.a_c0 = 0; e.b_k0 = 0; e.bmap = 0; e.b_z = (int16_t)(ky * d->ksize + kx);
        e.nchunks = (int16_t)(d->Cin / 64);
        if (merged) {
          e.amap = 0;
          e.b_z = (int16_t)(ph * 4 + ky * 2 + kx);
          e.d2 = (int16_t)((py == 0 ? -1 : 0) + ky);
          e.d1 = (int16_t)((px == 0 ? -1 : 0) + kx);
        } else if (d->upsample) {
          // source row = i + floor((py + ky - 1) / 2)
          int a = py + ky - pad, b = px + kx - pad;
          e.amap = 0;
          e.d2 = (int16_t)(a < 0 ? -1 : a / 2);
          e.d1 = (int16_t)(b < 0 ? -1 : b / 2);
        } else if (d->stride == 2) {
          // input row = 2*oy + ky - pad = 2*(oy + off) + phase
          int a = ky - pad, b = kx - pad;
          int pa = ((a % 2) + 2) % 2, pb = ((b % 2) + 2) % 2;
          e.amap = (int16_t)(pa * 2 + pb);
          e.d2 = (int16_t)((a - pa) / 2);
          e.d1 = (int16_t)((b - pb) / 2);
        } else {
          e.amap = 0; e.d2 = (int16_t)(ky - pad); e.d1 = (int16_t)(kx - pad);
        }
        kb += e.nchunks;
      }
    if (d->x2) {
      TcEntry& e = p.e[ne++];
      e.amap = 4; e.bmap = 1; e.a_c0 = 0; e.b_k0 = 0; e.b_z = 0; e.d1 = 0; e.d2 = 0;
      e.nchunks = (int16_t)(d->Cin2 / 64);
      kb += e.nchunks;
    }
    p.n_entries = ne; p.total_kb = kb;
    p.mul1 = d->upsample ? 2 : 1; p.mul2 = p.mul1;
    p.off1 = d->upsample ? px : 0; p.off2 = d->upsample ? py : 0;
    p.n_tiles = cdiv(d->Cout, bn);
    if (p.ksplit > 1) WSR_REQUIRE(kb == p.total_kb && (p.ksplit - 1) * p.kb_split < kb, WSR_E_INVALID, "conv_tc: split-K plan / K block count mismatch");
    g_last_ksplit = p.ksplit; g_last_bn = bn;
    switch (bn) {
      case 256: rc = launch_tc<256>(p, st); break;
      case 128: rc = launch_tc<128>(p, st); break;
      default: rc = launch_tc<64>(p, st); break;
    }
    if (rc) return rc;
  }
  if (d->gn_stats && !fuse_stats)
    return wsr_gn_stats(d->y, d->y_dtype, d->N, OH * OW, d->Cout, d->y_ld, d->gn_stats, d->gn_stats_ld, stream);
  return WSR_OK;
}

// 1 when wsr_conv_tc would run this descriptor in halo mode, i.e. can take a fused GroupNorm input (gn_table)
extern "C" int wsr_conv_tc_can_fuse_gn(const WsrConvDesc* d) {
  if (d == nullptr || d->x_dtype != WSR_BF16 || d->ksize != 3 || d->stride != 1 || d->upsample != 0) return 0;
  if (d->Cin % 64 != 0 || (d->x2 && d->Cin2 % 64 != 0)) return 0;
  int t1, t2, t3;
  choose_tile(d->W, d->H, d->N, t1, t2, t3);
  return (t2 == 1 && t3 == 1 && t1 + 2 <= 130) ? 1 : 0;
}

// Tap-table variant (data gradients of the stride-2 / upsample convolutions; see wsr.h).  Classic (non-halo) tiles only.
extern "C" int wsr_conv_taps_tc(const WsrConvDesc* d, const WsrTapTable* t, void* stream) {
  int rc = validate_conv_desc(d);
  if (rc) return rc;
  rc = validate_taps(t);
  if (rc) return rc;
  WSR_REQUIRE(t->in_sub <= 2, WSR_E_UNSUPPORTED, "conv_taps_tc: in_sub=%d (1 or 2)", t->in_sub);
  WSR_REQUIRE(d->x_dtype == WSR_BF16, WSR_E_UNSUPPORTED, "conv_taps_tc: bf16 operands only");
  WSR_REQUIRE(d->Cin % 64 == 0 && d->x_ld % 8 == 0 && (((uintptr_t)d->x) & 15) == 0 && (((uintptr_t)d->w) & 15) == 0,
              WSR_E_UNSUPPORTED, "conv_taps_tc: Cin %% 64, pitch %% 8 and 16-byte alignment required (Cin=%d ld=%d)", d->Cin, d->x_ld);
  WSR_REQUIRE(d->x2 == nullptr, WSR_E_UNSUPPORTED, "conv_taps_tc: no second segment");
  WSR_REQUIRE((((uintptr_t)d->bias) & 15) == 0 && (((uintptr_t)d->rowvec) & 15) == 0 && (d->rowvec == nullptr || d->rowvec_ld % 4 == 0),
              WSR_E_UNSUPPORTED, "conv_taps_tc: bias / rowvec must be 16-byte aligned, rowvec_ld %% 4 == 0");
  WSR_REQUIRE(t->in_sub == 1 || (d->H % 2 == 0 && d->W % 2 == 0), WSR_E_UNSUPPORTED, "conv_taps_tc: in_sub 2 needs even H, W");
  WSR_REQUIRE(d->gn_stats == nullptr || (t->out_mul == 1 && t->GH == t->OH && t->GW == t->OW), WSR_E_UNSUPPORTED,
              "conv_taps_tc: fused statistics need a launch that covers the whole output");
  cudaStream_t st = (cudaStream_t)stream;
  const int GH = t->GH, GW = t->GW, OH = t->OH, OW = t->OW;

  TcParams p;
  memset(&p, 0, sizeof(p));
  choose_tile(GW, GH, d->N, p.t1, p.t2, p.t3);
  WSR_REQUIRE(p.t1 <= 256 && p.t2 <= 256 && p.t3 <= 256, WSR_E_UNSUPPORTED, "conv_taps_tc: tile");
  p.g1 = cdiv(GW, p.t1); p.g2 = cdiv(GH, p.t2); p.g3 = cdiv(d->N, p.t3);
  p.nbatch = 1; p.a_zmul = 0; p.b_zmul = 0;
  p.a_bytes = p.t1 * p.t2 * p.t3 * 128;
  p.M1 = GW; p.M2 = GH; p.M3 = d->N;
  p.Ncols = d->Cout;
  p.out = d->y; p.out_dtype = d->y_dtype;
  p.o_s1 = d->y_ld; p.o_s2 = (long long)OW * d->y_ld; p.o_s3 = (long long)OH * OW * d->y_ld; p.o_sb = 0; p.o_sc = 1;
  p.bias = d->bias; p.rowvec = d->rowvec; p.rowvec_ld = d->rowvec_ld;
  p.act = d->act; p.out_scale = d->out_scale;
  p.res = d->res; p.res_dtype = d->res_dtype; p.res_scale = d->res_scale;
  p.r_s1 = d->res_ld; p.r_s2 = (long long)OW * d->res_ld; p.r_s3 = (long long)OH * OW * d->res_ld; p.r_sc = 1;
  p.res2 = d->res2; p.res2_dtype = d->res2_dtype; p.res2_scale = d->res2_scale;
  p.q_s1 = d->res2_ld; p.q_s2 = (long long)OW * d->res2_ld; p.q_s3 = (long long)OH * OW * d->res2_ld; p.q_sc = 1;
  const int m_tiles = p.g1 * p.g2 * p.g3;
  const int bn = pick_block_n(d->Cout, m_tiles);
  p.n_taps = 0; p.halo_rows = 1;
  p.ksplit = 1;
  if (stage_preconditions(p, bn)) {
    const int kb_est = t->ntaps * (d->Cin / 64);
    p.ksplit = pick_split(d->Cout, m_tiles, kb_est, bn);
    p.kb_split = cdiv(kb_est, p.ksplit);
  }
  const bool fuse_stats = d->gn_stats != nullptr && (p.t1 * p.t2) % 32 == 0;
  p.stats = fuse_stats ? d->gn_stats : nullptr;
  p.stats_ld = d->gn_stats_ld;

  int wt_count = 0;
  for (int i = 0; i < t->ntaps; ++i) if (t->wtap[i] + 1 > wt_count) wt_count = t->wtap[i] + 1;
  {
    const int wrows = d->w_rows > 0 ? d->w_rows : d->Cout;
    uint64_t dims[3] = {(uint64_t)d->Cin, (uint64_t)wrows, (uint64_t)wt_count};
    uint64_t str[2] = {(uint64_t)d->Cin * 2, (uint64_t)d->Cin * wrows * 2};
    uint32_t box[3] = {64, (uint32_t)bn, 1};
    rc = encode_map(&p.bmap[0], d->w, 3, dims, str, box);
    if (rc) return rc;
    p.bmap[1] = p.bmap[0];
  }
  const uint32_t abox[4] = {64, (uint32_t)p.t1, (uint32_t)p.t2, (uint32_t)p.t3};
  const long long ld = d->x_ld;
  if (t->in_sub == 1) {
    uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)d->W, (uint64_t)d->H, (uint64_t)d->N};
    uint64_t str[3] = {(uint64_t)ld * 2, (uint64_t)d->W * ld * 2, (uint64_t)d->H * d->W * ld * 2};
    rc = encode_map(&p.amap[0], d->x, 4, dims, str, abox);
    if (rc) return rc;
    for (int i = 1; i < kNumAMaps; ++i) p.amap[i] = p.amap[0];
  } else {
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)d->W / 2, (uint64_t)d->H / 2, (uint64_t)d->N};
        uint64_t str[3] = {(uint64_t)ld * 4, (uint64_t)d->W * ld * 4, (uint64_t)d->H * d->W * ld * 2};
        const __nv_bfloat16* base = (const __nv_bfloat16*)d->x + ((long long)py * d->W + px) * ld;
        rc = encode_map(&p.amap[py * 2 + px], base, 4, dims, str, abox);
        if (rc) return rc;
      }
    p.amap[4] = p.amap[0];
  }
  int kb = 0;
  for (int i = 0; i < t->ntaps; ++i) {
    TcEntry& e = p.e[i];
    e.amap = (int16_t)(t->in_sub == 2 ? t->py[i] * 2 + t->px[i] : 0);
    e.bmap = 0; e.a_c0 = 0; e.b_k0 = 0;
    e.b_z = (int16_t)t->wtap[i];
    e.d1 = (int16_t)t->dx[i]; e.d2 = (int16_t)t->dy[i];
    e.nchunks = (int16_t)(d->Cin / 64);
    kb += e.nchunks;
  }
  p.n_entries = t->ntaps; p.total_kb = kb;
  p.mul1 = t->out_mul; p.mul2 = t->out_mul; p.off1 = t->out_px; p.off2 = t->out_py;
  p.n_tiles = cdiv(d->Cout, bn);
  if (p.ksplit > 1) WSR_REQUIRE((p.ksplit - 1) * p.kb_split < kb, WSR_E_INVALID, "conv_taps_tc: split-K plan / K block count mismatch");
  g_last_ksplit = p.ksplit; g_last_bn = bn;
  switch (bn) {
    case 256: rc = launch_tc<256>(p, st); break;
    case 128: rc = launch_tc<128>(p, st); break;
    default: rc = launch_tc<64>(p, st); break;
  }
  if (rc) return rc;
  if (d->gn_stats && !fuse_stats)
    return wsr_gn_stats(d->y, d->y_dtype, d->N, OH * OW, d->Cout, d->y_ld, d->gn_stats, d->gn_stats_ld, stream);
  return WSR_OK;
}

extern "C" int wsr_gemm_tc(const WsrGemmDesc* g, void* stream) {
  int rc = validate_gemm_desc(g);
  if (rc) return rc;
  WSR_REQUIRE(g->a_dtype == WSR_BF16 && g->b_dtype == WSR_BF16, WSR_E_UNSUPPORTED, "gemm_tc: bf16 operands only");
  // operand majorness from the strides: unit k stride = K-major; unit row / column stride = MN-major (transposed operand)
  const bool a_mn = g->a_sk != 1, b_mn = g->b_sk != 1;
  WSR_REQUIRE(!a_mn || g->a_sm == 1, WSR_E_UNSUPPORTED, "gemm_tc: A needs a unit stride along k or along m");
  WSR_REQUIRE(!b_mn || g->b_sn == 1, WSR_E_UNSUPPORTED, "gemm_tc: B needs a unit stride along k or along n");
  WSR_REQUIRE(g->K % 64 == 0, WSR_E_UNSUPPORTED, "gemm_tc: K=%d must be a multiple of 64", g->K);
  WSR_REQUIRE((((uintptr_t)g->bias) & 15) == 0, WSR_E_UNSUPPORTED, "gemm_tc: bias must be 16-byte aligned");
  const int64_t a_pitch = a_mn ? g->a_sk : g->a_sm, b_pitch = b_mn ? g->b_sk : g->b_sn;
  WSR_REQUIRE(a_pitch % 8 == 0 && b_pitch % 8 == 0 && g->a_sb % 8 == 0 && g->b_sb % 8 == 0 && (((uintptr_t)g->a) & 15) == 0 &&
                  (((uintptr_t)g->b) & 15) == 0,
              WSR_E_UNSUPPORTED, "gemm_tc: strides must be multiples of 8 elements, bases 16-byte aligned");
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.t1 = g->M < 128 ? g->M : 128; p.t2 = 1; p.t3 = 1;
  p.g1 = cdiv(g->M, p.t1); p.g2 = 1; p.g3 = 1;
  p.nbatch = g->batch; p.a_zmul = 1; p.b_zmul = 1;
  p.a_mn = a_mn ? 1 : 0; p.b_mn = b_mn ? 1 : 0;
  p.a_blk = cdiv(p.t1, 64);
  p.a_bytes = a_mn ? p.a_blk * 8192 : p.t1 * 128;
  p.M1 = g->M; p.M2 = 1; p.M3 = 1;
  p.Ncols = g->N;
  p.out = g->d; p.out_dtype = g->d_dtype;
  p.o_s1 = g->d_sm; p.o_s2 = 0; p.o_s3 = 0; p.o_sb = g->d_sb; p.o_sc = g->d_sn;
  p.mul1 = 1; p.mul2 = 1;
  p.bias = g->bias; p.act = WSR_ACT_NONE; p.out_scale = g->alpha;
  p.res = g->res; p.res_dtype = g->res_dtype; p.res_scale = 1.f;
  p.r_s1 = g->res_sm; p.r_sb = g->res_sb; p.r_sc = g->res_sn;
  const int m_tiles = p.g1 * g->batch;
  const int bn = pick_block_n(g->N, m_tiles);
  p.b_blk = cdiv(bn < g->N ? bn : g->N, 64);
  p.b_bytes = b_mn ? p.b_blk * 8192 : 0;
  {
    uint64_t dims[4], str[3];
    uint32_t box[4];
    if (!a_mn) {
      dims[0] = (uint64_t)g->K; dims[1] = (uint64_t)g->M; dims[2] = 1; dims[3] = (uint64_t)g->batch;
      str[0] = (uint64_t)g->a_sm * 2; str[1] = (uint64_t)g->a_sm * g->M * 2; str[2] = (uint64_t)(g->batch > 1 ? g->a_sb : g->a_sm * g->M) * 2;
      box[0] = 64; box[1] = (uint32_t)p.t1; box[2] = 1; box[3] = 1;
    } else {
      dims[0] = (uint64_t)g->M; dims[1] = (uint64_t)g->K; dims[2] = 1; dims[3] = (uint64_t)g->batch;
      str[0] = (uint64_t)g->a_sk * 2; str[1] = (uint64_t)g->a_sk * g->K * 2; str[2] = (uint64_t)(g->batch > 1 ? g->a_sb : g->a_sk * g->K) * 2;
      box[0] = 64; box[1] = 64; box[2] = 1; box[3] = 1;
    }
    if (g->batch > 1 && g->a_sb == 0) { dims[3] = 1; p.a_zmul = 0; str[2] = str[1]; }
    rc = encode_map(&p.amap[0], g->a, 4, dims, str, box);
    if (rc) return rc;
    for (int i = 1; i < kNumAMaps; ++i) p.amap[i] = p.amap[0];
  }
  {
    uint64_t dims[3], str[2];
    uint32_t box[3];
    if (!b_mn) {
      dims[0] = (uint64_t)g->K; dims[1] = (uint64_t)g->N; dims[2] = (uint64_t)g->batch;
      str[0] = (uint64_t)g->b_sn * 2; str[1] = (uint64_t)(g->batch > 1 ? g->b_sb : g->b_sn * g->N) * 2;
      box[0] = 64; box[1] = (uint32_t)bn; box[2] = 1;
      if (g->batch > 1 && g->b_sb == 0) { dims[2] = 1; p.b_zmul = 0; str[1] = (uint64_t)g->b_sn * g->N * 2; }
    } else {
      dims[0] = (uint64_t)g->N; dims[1] = (uint64_t)g->K; dims[2] = (uint64_t)g->batch;
      str[0] = (uint64_t)g->b_sk * 2; str[1] = (uint64_t)(g->batch > 1 ? g->b_sb : g->b_sk * g->K) * 2;
      box[0] = 64; box[1] = 64; box[2] = 1;
      if (g->batch > 1 && g->b_sb == 0) { dims[2] = 1; p.b_zmul = 0; str[1] = (uint64_t)g->b_sk * g->K * 2; }
    }
    rc = encode_map(&p.bmap[0], g->b, 3, dims, str, box);
    if (rc) return rc;
    p.bmap[1] = p.bmap[0];
  }
  p.n_entries = 1;
  p.e[0].amap = 0; p.e[0].bmap = 0; p.e[0].a_c0 = 0; p.e[0].b_k0 = 0; p.e[0].b_z = 0; p.e[0].d1 = 0; p.e[0].d2 = 0;
  WSR_REQUIRE(g->K / 64 <= 32767, WSR_E_UNSUPPORTED, "gemm_tc: K too large");
  p.e[0].nchunks = (int16_t)(g->K / 64);
  p.total_kb = g->K / 64;
  p.n_tiles = cdiv(g->N, bn);
  cudaStream_t st = (cudaStream_t)stream;
  switch (bn) {
    case 256: return launch_tc<256>(p, st);
    case 128: return launch_tc<128>(p, st);
    default: return launch_tc<64>(p, st);
  }
}
