// 3^3 stride-1 Conv3D, persistent halo-reuse kernel (the hot conv of the U-Net and decoders).
//
// Why: with one TMA tile per (tap, chunk) the 27 taps re-fetch the same voxels 27x.  Here each CTA stages HALO SLABS
// once and re-uses them:
//
//   tile      8 w x 16 h x TD d output voxels (TD accumulators of M=128 in TMEM), BLOCK_N output channels
//   slab      one input d-plane of the halo: 10 w x 18 h voxels x 64 channels, one 5-D TMA box {64,10,18,1,1} with
//             SWIZZLE_128B (23040 B; 'same' padding = TMA out-of-bounds zero fill).  A slab serves the 9 in-plane taps
//             of up to 3 (kd) x TD (plane) accumulations: the (kh,kw) shift is applied by moving the UMMA
//             descriptor start by (kh*10+kw) 128-B rows with SBO = 10 rows -- legal because SWIZZLE_128B addressing
//             is a pure function of the absolute smem address (verified on B200; base_offset stays 0).
//   slab ring NS slabs; taps run kd-major so slab 0 is released after kd=0, slab 1 after kd=1, the rest after kd=2,
//             and the next chunk's / next tile's slabs stream in behind them.
//   B ring    TPS taps (one kh row: kw = 0..2) of [BLOCK_N x 64] weights per stage, one 3-D TMA box {64,BLOCK_N,TPS};
//             shared by the TD planes -> TPS*TD*4 MMAs per barrier round trip.  Measured on B200 (tools/issue_probe.cu):
//             an mbarrier wait costs ~110 cycles and a commit ~45 on the single issuing thread, and an M128xN64xK16
//             MMA only 48, so one tap per round trip is issue-bound; three are not.
//   TMEM      2 accumulator stages x TD x BLOCK_N columns: the epilogue of tile i overlaps the MMAs of tile i+1.
//   shortcut  optional 1^3 conv of two more tensors (mapS0 / mapS1: a ResidualBlock's [x | skip]) in the same accumulators, after
//             the 3^3 chunks: per 64-channel chunk TD slabs (pair: the kd = 1 pair slab) of the same halo box, read at the
//             centre tap only; its k-blocks follow the 3^3 ones in the weight rows (one tap each, padded to whole stages).
//
// Warps (384 threads): 0 = slab producer, 1 = weight producer, 2 = TMEM owner + MMA issuer, 3 = second MMA issuer (TD = 2), 4-11 = epilogue.
// Every role loop is warp-uniform; a single elected lane (elect.sync) issues TMA / tcgen05 instructions.
#pragma once
#include "conv_common.cuh"

namespace halo {

constexpr int kThreads = 384;
constexpr int kThreadsFused = 416;         // FUSE_UPD: + one warp that owns the epilogue's TMA traffic (see the kernel)
constexpr int kSlabBytes = 23 * 1024;      // 180 voxels x 128 B = 23040, rounded up to the 1024-B swizzle period
constexpr int kSlabTx = 180 * 128;

struct Tile {
  int w0, h0, d0, n, n_tile;
};

template <bool PAIR = false>
__device__ __forceinline__ Tile decode_tile(const ConvParams& p, int id) {
  Tile t;
  t.n_tile = id / p.halo_tiles_per_ntile;
  int r = id - t.n_tile * p.halo_tiles_per_ntile;
  t.w0 = (r % p.tiles_w) * 8; r /= p.tiles_w;
  t.h0 = (r % p.tiles_h) * (PAIR ? 8 : 16); r /= p.tiles_h;
  t.d0 = (r % p.tiles_d) * p.halo_td; r /= p.tiles_d;
  t.n = r;
  return t;
}

// staged epilogue: output staging buffers (each holds one plane's BLOCK_N/64 column groups of 128 rows x 128 B)
constexpr int stage_bufs(int block_n) { return block_n <= 64 ? 2 : 1; }
constexpr int stage_groups(int block_n) { return block_n >= 64 ? block_n / 64 : 1; }          // 64-channel groups (one 32-channel group)
constexpr int stage_group_bytes(int block_n) { return block_n >= 64 ? 16384 : 8192; }         // 128 rows x 128 B | x 64 B
constexpr int kFuseStage16Bytes = 2 * 8192;
constexpr int stage_bytes(int block_n, bool staged) { return staged ? stage_bufs(block_n) * stage_groups(block_n) * stage_group_bytes(block_n) : 0; }

// Shared-memory layout of conv_halo_kernel and conv_halo_up_kernel (TPS = 4, CG2, STAGED), offsets from the 1024-aligned base:
// slab ring | weight ring | output staging | FUSE_UPD 16-bit staging | barriers | TMEM address | bias + scale [2][2][BLOCK_N].
template <int BLOCK_N, int NS, int NB, int TPS, bool STAGED, bool PAIR, bool CG2, bool FUSE_UPD>
struct Smem {
  static constexpr int kSlabBytes = PAIR ? 25 * 1024 : halo::kSlabBytes;   // 200 (pair) / 180 rows of 128 B, 1 KB-rounded
  static constexpr int kBRows = CG2 ? BLOCK_N / 2 : BLOCK_N;               // weight rows of one tap staged by THIS CTA
  static constexpr int kTapBytes = kBRows * 128;
  static constexpr int kBBytes = TPS * kTapBytes;                           // one weight stage
  // slab full / empty, weight full / empty, TMEM full / empty x 2; FUSE_UPD: + x_t landed / tiles written x 2 staging sets
  static constexpr int kBars = 2 * NS + 2 * NB + 4 + (FUSE_UPD ? 4 : 0);
  static constexpr size_t kBRing = (size_t)NS * kSlabBytes;
  static constexpr size_t kStage = kBRing + (size_t)NB * kBBytes;          // (1024-aligned: slabs and weight stages are multiples of 1 KB)
  static constexpr size_t kStage16 = kStage + stage_bytes(BLOCK_N, STAGED);
  static constexpr size_t kBarOff = kStage16 + (FUSE_UPD ? kFuseStage16Bytes : 0);
  static constexpr size_t kTmemPtr = kBarOff + (size_t)kBars * 8;
  static constexpr size_t kBias = kTmemPtr + 16;
  static constexpr size_t kBytes = 1024 + kBias + 4 * BLOCK_N * 4;         // with the alignment slack
};

// ---------------------------------------------------------------- pieces shared by conv_halo_kernel and conv_halo_up_kernel

// Barriers from the base of the barrier area: slab full / empty [NS], weight full / empty [NB], accumulator (TMEM) full / empty [2].
template <int NS, int NB>
struct Bars {
  uint32_t base;
  __device__ __forceinline__ uint32_t slab_full(int s) const { return base + 8u * s; }
  __device__ __forceinline__ uint32_t slab_empty(int s) const { return base + 8u * (NS + s); }
  __device__ __forceinline__ uint32_t b_full(int s) const { return base + 8u * (2 * NS + s); }
  __device__ __forceinline__ uint32_t b_empty(int s) const { return base + 8u * (2 * NS + NB + s); }
  __device__ __forceinline__ uint32_t tmem_full(int s) const { return base + 8u * (2 * NS + 2 * NB + s); }
  __device__ __forceinline__ uint32_t tmem_empty(int s) const { return base + 8u * (2 * NS + 2 * NB + 2 + s); }
  // (thread 0) `issuers`: arrivals that release a slab / weight stage and fill an accumulator stage; `releasers`: arrivals
  // that hand an accumulator stage back
  __device__ __forceinline__ void init(uint32_t issuers, uint32_t releasers) const {
    for (int s = 0; s < NS; ++s) { ptx::mbar_init(slab_full(s), 1); ptx::mbar_init(slab_empty(s), issuers); }
    for (int s = 0; s < NB; ++s) { ptx::mbar_init(b_full(s), 1); ptx::mbar_init(b_empty(s), issuers); }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(tmem_full(s), issuers); ptx::mbar_init(tmem_empty(s), releasers); }
  }
};

// TMEM allocation by warp 2 (of both CTAs under CG2), permit relinquished at once
template <bool CG2>
__device__ __forceinline__ void tmem_alloc(uint32_t* tmem_ptr_smem, uint32_t cols) {
  if (CG2) { ptx::tmem_alloc_cg2(ptx::smem_u32(tmem_ptr_smem), cols); ptx::tmem_relinquish_cg2(); }
  else { ptx::tmem_alloc(ptx::smem_u32(tmem_ptr_smem), cols); ptx::tmem_relinquish(); }
}

// End of the set-up: every thread sees the barriers and the TMEM address (CG2: the peer's barriers exist -- fence_barrier_init --
// before anything signals them); then wait for the previous kernel, whose tail the set-up overlapped.  Returns the TMEM base.
template <bool CG2>
__device__ __forceinline__ uint32_t setup_join(const uint32_t* tmem_ptr_smem) {
  ptx::tc_fence_before();
  __syncthreads();
  if (CG2) ptx::cluster_sync_exit();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();
  return tmem_base;
}

// Kernel tail: all roles are done; under CG2 the leader's MMAs read the peer's shared memory / write its TMEM until the cluster
// barrier.  Warp 2 frees the TMEM.  `tp`: the launch's parameters when the tail is traced (timeline region 3), else nullptr.
template <bool CG2>
__device__ __forceinline__ void teardown(const ConvParams* tp, uint32_t tmem_base, uint32_t cols) {
  int tx = 0;
  if (tp && threadIdx.x == 128) trace_ev(*tp, 3, tx, 30);
  ptx::tc_fence_before();
  __syncthreads();
  if (tp && threadIdx.x == 128) trace_ev(*tp, 3, tx, 31);
  if (CG2) ptx::cluster_sync_exit();
  if (tp && threadIdx.x == 128) trace_ev(*tp, 3, tx, 32);
  if ((threadIdx.x >> 5) == 2) {
    ptx::tc_fence_after();
    if (CG2) ptx::tmem_dealloc_cg2(tmem_base, cols); else ptx::tmem_dealloc(tmem_base, cols);
  }
}

// The MMA issuer's position in the slab ring: qs = slot of the current chunk's first slab, qph = its phase bit.  Carried
// incrementally: the issuing thread is the pacing resource, and the integer divisions / modulos of a closed-form index cost
// ~200 cycles per kd step during which the shallow MMA queue drains.
template <int NS>
struct SlabCursor {
  uint32_t qs = 0, qph = 0;
  __device__ __forceinline__ uint32_t slot(uint32_t i, uint32_t& ph) const {   // ring slot / phase of slab i of the chunk (i < NS)
    uint32_t idx = qs + i;
    const bool wrap = idx >= (uint32_t)NS;
    ph = qph ^ (wrap ? 1u : 0u);
    return wrap ? idx - NS : idx;
  }
  __device__ __forceinline__ void advance(uint32_t k) {
    qs += k;
    if (qs >= (uint32_t)NS) { qs -= NS; qph ^= 1; }
  }
};

// Weight producer (warp 1): per tile, `stages` weight stages of `kps` consecutive k-blocks (the box depth of mapB) from weight
// row row_of(tile id), for the tiles first_tile, first_tile + tile_step, ... (the kernel's schedule); under CG2 each CTA loads
// its kBRows rows of the stage, completing on the leader's barrier.
template <int NS, int NB, int kBRows, int kBBytes, bool CG2, class RowOf>
__device__ __forceinline__ void produce_weights(const ConvParams& p, const Bars<NS, NB>& bar, const CUtensorMap* mapB, uint32_t bring_base,
                                                uint32_t crank, int first_tile, int tile_step, int stages, int kps, int dbg_code,
                                                RowOf&& row_of) {
  uint32_t s = 0, ph = 1;
  bool ok = true;
  for (int id = first_tile; id < p.halo_total_tiles && ok; id += tile_step) {
    const int row0 = row_of(id);
    for (int kb = 0; kb < stages * kps; kb += kps) {
      ok = ptx::mbar_wait(bar.b_empty(s), ph, p.dbg, dbg_code);
      if (!ok) break;
      if (ptx::elect_one()) {
        if (CG2) {
          if (crank == 0) ptx::mbar_expect_tx(bar.b_full(s), 2 * kBBytes);
          ptx::tma_load_3d_cg2(bring_base + s * kBBytes, mapB, ptx::mapa_shared(bar.b_full(s), 0), 0, row0 + (int)crank * kBRows, kb);
        } else {
          ptx::mbar_expect_tx(bar.b_full(s), kBBytes);
          ptx::tma_load_3d(bring_base + s * kBBytes, mapB, bar.b_full(s), 0, row0, kb);
        }
      }
      __syncwarp();
      if (++s == NB) { s = 0; ph ^= 1; }
    }
  }
}

// Bias + temb row of sample n for the tile's BLOCK_N columns from col_base -> bs / scs (the buffer of the tile's accumulator
// stage), by the 256 epilogue threads BEFORE the accumulator is ready: the two dependent global round trips (t_dev, then the
// table rows: ~1.5 k cycles) overlap the tile's MMAs instead of heading its epilogue.  The buffer was last read in tile it - 2;
// every epilogue thread has passed a bar.sync of tile it - 1 since.  `ti`: the epilogue's trace index (event 20), or nullptr.
template <int BLOCK_N>
__device__ __forceinline__ void stage_tile_bias(const ConvParams& p, float* bs, float* scs, int n, int col_base, int* ti) {
  const float* cbrow = nullptr;
  if (p.chan_bias) {
    const int tt = p.t_dev ? p.t_dev[0] : 0;
    cbrow = p.chan_bias + ((int64_t)tt * p.chan_bias_rows + (p.chan_bias_rows > 1 ? n : 0)) * p.c_out;
  }
  stage_bias(p, bs, scs, col_base, BLOCK_N, cbrow, threadIdx.x - 128, 256);
  if (ti && threadIdx.x == 128) trace_ev(p, 1, *ti, 20);
  epilogue_bar_sync256();
}

// Staged 16-bit store of one output plane: wait until the staging buffer nstore % kBufs is free, run this thread's row of
// TMEM columns [taddr, + BLOCK_N / 2) through conv_epilogue16_staged into it (whole 128-byte rows, SWIZZLE_128B; BLOCK_N = 32:
// 64-byte rows, SWIZZLE_64B), then one TMA store per 64-channel group at (col_base + 64 g, w0, h0, od, n) -- PAIR: (.., w0, od,
// h0, n) -- with the edges clipped by the TMA unit (row-per-thread 16-byte stores touch 32 lines per instruction).
// bs / scs: the tile's staged bias and scale (used when has_bs / has_sc); `rpre`: this plane's residual rows in registers
// (kChunks x 2 vectors), or nullptr; `ti`: the epilogue's trace index (events 13-15), or nullptr.
template <int BLOCK_N, bool PAIR>
__device__ __forceinline__ void store_plane16(const ConvParams& p, const CUtensorMap* map, uint8_t* stg_base, uint32_t nstore,
                                              uint32_t taddr, int r, int cbase, int col_base, const float* bs, const float* scs,
                                              bool has_bs, bool has_sc, int w0, int h0, int od, int n, bool pre,
                                              const bf16x8 (*rpre)[2], int* ti) {
  constexpr int kChunks = BLOCK_N / 32;   // 16-column chunks of this warp's column half
  constexpr int kNG = stage_groups(BLOCK_N), kBufs = stage_bufs(BLOCK_N), kGB = stage_group_bytes(BLOCK_N);
  constexpr bool kRow64 = BLOCK_N < 64;   // one 32-channel group: 64-byte rows, SWIZZLE_64B
  const int grp = kRow64 ? 0 : cbase >> 6, cl0 = kRow64 ? cbase : cbase & 63;
  const bool ev = ti && threadIdx.x == 128;
  const int colt = col_base + cbase;
  uint8_t* stg = stg_base + ((nstore % kBufs) * kNG + grp) * kGB;
  if (threadIdx.x == 128) {   // the store that last used this buffer has finished reading it
    if (kBufs == 2) ptx::bulk_wait_read_1(); else ptx::bulk_wait_read_all();
  }
  epilogue_bar_sync256();
  if (ev) trace_ev(p, 1, *ti, 13);
#pragma unroll
  for (int c = 0; c < kChunks; c += 2) {
    const int col0 = colt + c * 16;
    uint32_t ra[16], rb[16];
    ptx::tc_ld_32x32b_x16(taddr + c * 16, ra);
    if (c + 1 < kChunks) ptx::tc_ld_32x32b_x16(taddr + c * 16 + 16, rb);
    ptx::tc_wait_ld();
    conv_epilogue16_staged(p, ra, r, cl0 + c * 16, col0, has_bs ? bs + cbase + c * 16 : nullptr, nullptr,
                           has_sc ? scs + cbase + c * 16 : nullptr, nullptr, stg, pre, rpre ? rpre[c] : nullptr, kRow64);
    if (c + 1 < kChunks)
      conv_epilogue16_staged(p, rb, r, cl0 + c * 16 + 16, col0 + 16, has_bs ? bs + cbase + c * 16 + 16 : nullptr, nullptr,
                             has_sc ? scs + cbase + c * 16 + 16 : nullptr, nullptr, stg, pre,
                             rpre ? rpre[c + 1 < kChunks ? c + 1 : c] : nullptr, kRow64);
  }
  if (ev) trace_ev(p, 1, *ti, 14);
  ptx::fence_proxy_async();
  epilogue_bar_sync256();
  if (ev) trace_ev(p, 1, *ti, 15);
  if (threadIdx.x == 128) {
    for (int g = 0; g < kNG; ++g)
      if (col_base + g * 64 < p.c_out) {
        const uint32_t src = ptx::smem_u32(stg_base + ((nstore % kBufs) * kNG + g) * kGB);
        if (PAIR) ptx::tma_store_5d(map, src, col_base + g * 64, w0, od, h0, n);
        else ptx::tma_store_5d(map, src, col_base + g * 64, w0, h0, od, n);
      }
    ptx::bulk_commit_group();
  }
}

// Hand accumulator stage `as` back to the (leader's) MMA issuers, by lane 0 of each epilogue warp -- only for a tile that has a
// successor two tiles on: nobody ever waits for the arrivals of a CTA's last two tiles, and the cluster-scope arrive costs the
// arriving warp 2-2.5 k cycles (clock64 timeline) -- on the one-tile CTAs of the 16^3 / 8^3 levels that was the tail of a fully
// exposed epilogue.
template <bool CG2>
__device__ __forceinline__ void release_acc(const ConvParams& p, uint32_t tmem_empty, int id, int tile_step) {
  if ((threadIdx.x & 31) == 0 && id + 2 * tile_step < p.halo_total_tiles) {
    if (CG2) ptx::mbar_arrive_cluster(ptx::mapa_shared(tmem_empty, 0));
    else ptx::mbar_arrive(tmem_empty);
  }
}

// PAIR (small planes, 8 x 8: the 8^3 level of the U-Net): the tile is 8 w x 8 h x 2 d.  The activation tensor map lists
// its dims as (C, W, D, H, N), so one box {64, 10, 2, 10, 1} lands in smem as rows [h][d][w]: the 16 eight-row groups of
// the M = 128 operand (group = h * 2 + d) are again a uniform 10 rows apart, the (kh, kw) tap shift is (kh * 20 + kw) rows,
// and each kd tap reads its own pair slab (planes d0 + kd - 1, d0 + kd).  TD = 1; staged epilogue only.
// CG2 (cta_group::2): a cluster of two CTAs works on two consecutive tiles of the same n-tile.  Each CTA stages its own slabs
// and HALF of every weight stage (BLOCK_N / 2 rows); the leader's issuer warps run M = 256 MMAs over both CTAs' shared memory
// and TMEM.  Per CTA and MMA that is 4 KB of A + 1 KB of B instead of 4 + 2, and half the weight fill traffic -- the two terms
// that put the one-CTA main loop on the shared-memory roofline.
// FUSE_UPD (BLOCK_N = 128, fp32 staged output: the U-Net's eps conv on the sampling graph): the epilogue applies the
// reverse-diffusion update to its tile -- see ConvParams::upd_x.  mapY then addresses x_{t-1} (fp32) and mapZ its 16-bit copy.
template <int BLOCK_N, int TD, int NS, int NB, int TPS, bool STAGED, bool PAIR = false, bool CG2 = false, bool FUSE_UPD = false>
__global__ void __launch_bounds__(FUSE_UPD ? kThreadsFused : kThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                 const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapY,
                 const __grid_constant__ CUtensorMap mapZ, const __grid_constant__ CUtensorMap mapS0,
                 const __grid_constant__ CUtensorMap mapS1, const ConvParams p) {
  static_assert(!FUSE_UPD || (STAGED && BLOCK_N == 128 && !PAIR), "fused update: fp32 staged epilogue of the N = 128 tiles");
  static_assert(!STAGED || BLOCK_N >= 32, "staged epilogue works on whole 64-channel groups (or one 32-channel group)");
  static_assert(TPS == 1 || TPS == 3, "taps per weight stage: 1 or 3");
  static_assert(!PAIR || (STAGED && TD == 1), "pair-slab tiles: one accumulator, staged epilogue");
  using L = Smem<BLOCK_N, NS, NB, TPS, STAGED, PAIR, CG2, FUSE_UPD>;
  constexpr int kSlabBytes = L::kSlabBytes;
  constexpr int kSlabTx = PAIR ? 200 * 128 : halo::kSlabTx;
  constexpr int kKhUnits = PAIR ? 160 : 80;                          // one kh step in 16-byte units (20 / 10 rows)
  static_assert(!CG2 || BLOCK_N >= 32, "CTA-pair variant: each CTA stages BLOCK_N / 2 >= 16 weight rows");
  constexpr int kBRows = L::kBRows;
  constexpr int kTapBytes = L::kTapBytes;
  constexpr int kBBytes = L::kBBytes;
  // MMA issuer warps: with TD = 2 each output plane (its own TMEM accumulator) is driven by its own warp.  Measured
  // (clock64 timeline): one issuing thread spends ~280 cycles per weight stage on barrier waits / commits / descriptor
  // arithmetic during which the shallow tcgen05 queue drains (59 cycles per N=64 MMA instead of the 48-cycle floor);
  // two independent issuers hide each other's bookkeeping.
  constexpr int kIssuers = TD == 2 ? 2 : 1;
  constexpr uint32_t kAccCols = TD * BLOCK_N;
  constexpr uint32_t kTmemCols = (2 * kAccCols) < 32 ? 32 : 2 * kAccCols;
  static_assert(kTmemCols <= 512 && (kTmemCols & (kTmemCols - 1)) == 0, "TMEM columns must be a power of two <= 512");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* b_ring = smem + L::kBRing;
  uint8_t* stg_base = smem + L::kStage;
  uint8_t* stg16_base = smem + L::kStage16;   // FUSE_UPD: two 8 KB tiles (128 rows x 32 x 16 bit)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + L::kTmemPtr);
  float* bias_s = reinterpret_cast<float*>(smem + L::kBias);   // [2 acc stages][bias | scale][BLOCK_N]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t slab_base = ptx::smem_u32(smem);
  const uint32_t bring_base = ptx::smem_u32(b_ring);
  const uint32_t bar_base = ptx::smem_u32(bars);
  const Bars<NS, NB> bar{bar_base};
  auto x_bar = [&](uint32_t set) { return bar_base + 8u * (2 * NS + 2 * NB + 4 + 2 * set); };   // FUSE_UPD: the x_t tiles of staging set `set` have landed
  // FUSE_UPD: the 256 epilogue threads have written the tiles of staging set `set`.  One barrier PER SET: the writers only arrive
  // (they never wait on it), so a fast warp may arrive for round r + 1 before a slow warp has arrived for round r -- on a single
  // barrier that second arrival would be counted into round r's phase (seen as x_bar time-outs at batch 1: phases slipped).
  // Round r + 2 reuses round r's barrier, but nobody gets there before the agent has seen round r complete (x_bar[set]).
  auto w_bar = [&](uint32_t set) { return bar_base + 8u * (2 * NS + 2 * NB + 5 + 2 * set); };

  pdl_launch_dependents();
  const int nch = p.nch0 + p.nch1;
  const int sc_nch = p.sc_nch0 + p.sc_nch1;
  const int first_tile = blockIdx.x, tile_step = gridDim.x;
  const uint32_t crank = CG2 ? ptx::cluster_ctarank() : 0u;
  const bool leader = crank == 0;

  if (threadIdx.x == 0) {
    // accumulator-stage release: one arrival per epilogue warp (both CTAs of a pair); FUSE_UPD: one per CTA, by the TMA agent
    bar.init(kIssuers, FUSE_UPD ? (CG2 ? 2 : 1) : (CG2 ? 16 : 8));
    if (FUSE_UPD) { ptx::mbar_init(x_bar(0), 4); ptx::mbar_init(x_bar(1), 4); ptx::mbar_init(w_bar(0), 256); ptx::mbar_init(w_bar(1), 256); }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&mapA0);
    ptx::prefetch_tmap(&mapB);
    if (sc_nch > 0) ptx::prefetch_tmap(&mapS0);
    if (STAGED) ptx::prefetch_tmap(&mapY);
    if (FUSE_UPD) ptx::prefetch_tmap(&mapZ);
  }
  if (warp == 2) tmem_alloc<CG2>(tmem_ptr_smem, kTmemCols);
  const uint32_t tmem_base = setup_join<CG2>(tmem_ptr_smem);

  if (warp == 0) {
    // ===================== slab producer =====================
    uint32_t s = 0, ph = 1;
    bool ok = true;
    int ti = 0;
    // the next ring slot <- the slab of channels c0.. whose first input plane is d (pair slab: planes d, d + 1)
    auto load_slab = [&](const Tile& t, const CUtensorMap* map, int c0, int d, int tag) {
      ok = ptx::mbar_wait(bar.slab_empty(s), ph, p.dbg, 11);
      if (!ok) return;
      if (lane == 0) trace_ev(p, 2, ti, tag);
      if (ptx::elect_one()) {
        if (CG2) {   // both CTAs' slabs complete on the LEADER's barrier, which expects both transfers
          if (leader) ptx::mbar_expect_tx(bar.slab_full(s), 2 * kSlabTx);
          if (PAIR) ptx::tma_load_5d_cg2(slab_base + s * kSlabBytes, map, ptx::mapa_shared(bar.slab_full(s), 0), c0, t.w0 - 1, d, t.h0 - 1, t.n);
          else ptx::tma_load_5d_cg2(slab_base + s * kSlabBytes, map, ptx::mapa_shared(bar.slab_full(s), 0), c0, t.w0 - 1, t.h0 - 1, d, t.n);
        } else {
          ptx::mbar_expect_tx(bar.slab_full(s), kSlabTx);
          if (PAIR) ptx::tma_load_5d(slab_base + s * kSlabBytes, map, bar.slab_full(s), c0, t.w0 - 1, d, t.h0 - 1, t.n);
          else ptx::tma_load_5d(slab_base + s * kSlabBytes, map, bar.slab_full(s), c0, t.w0 - 1, t.h0 - 1, d, t.n);
        }
      }
      __syncwarp();
      if (++s == NS) { s = 0; ph ^= 1; }
    };
    for (int id = first_tile; id < p.halo_total_tiles && ok; id += tile_step) {
      const Tile t = decode_tile<PAIR>(p, id);
      for (int j = 0; j < nch && ok; ++j) {
        const CUtensorMap* map = j < p.nch0 ? &mapA0 : &mapA1;
        const int c0 = (j < p.nch0 ? j : j - p.nch0) * 64;
        for (int pl = 0; pl < TD + 2 && ok; ++pl) load_slab(t, map, c0, t.d0 - 1 + pl, 20 + pl);
      }
      // shortcut: the output planes themselves (pair: the kd = 1 slab)
      for (int j = 0; j < sc_nch && ok; ++j) {
        const CUtensorMap* map = j < p.sc_nch0 ? &mapS0 : &mapS1;
        const int c0 = (j < p.sc_nch0 ? j : j - p.sc_nch0) * 64;
        for (int pl = 0; pl < TD && ok; ++pl) load_slab(t, map, c0, t.d0 + pl, 24 + pl);
      }
    }
  } else if (warp == 1) {
    // ===================== weight producer: TPS taps per stage, the shortcut's k-blocks padded to whole stages =====================
    produce_weights<NS, NB, kBRows, kBBytes, CG2>(p, bar, &mapB, bring_base, crank, first_tile, tile_step, nch * 27 / TPS + (sc_nch + TPS - 1) / TPS, TPS, 12,
                                                  [&](int id) { return decode_tile<PAIR>(p, id).n_tile * BLOCK_N; });
  } else if (warp == 2 || (warp == 3 && kIssuers == 2)) {
    // ===================== MMA issuer(s) =====================
    const int pl_lo = kIssuers == 2 ? warp - 2 : 0, pl_hi = kIssuers == 2 ? warp - 1 : TD;   // planes this warp drives
    const bool tr = warp == 2;   // (only the elected lane runs the loop below)
    // Descriptors are formed by ADDING 16-byte units to precomputed 64-bit bases (the 14-bit address field cannot
    // carry: smem < 256 KB); inside a stage every offset is a compile-time immediate.
    constexpr uint32_t idesc = ptx::make_idesc_act(CG2 ? 256 : 128, BLOCK_N);
    auto mma = [&](uint32_t d, uint64_t da, uint64_t db, uint32_t accum) {
      if (CG2) ptx::tc_mma_f16_cg2(d, da, db, idesc, accum); else ptx::tc_mma_f16(d, da, db, idesc, accum);
    };
    auto commit = [&](uint32_t bar) { if (CG2) ptx::tc_commit_cg2(bar, (uint16_t)3); else ptx::tc_commit(bar); };
    const uint64_t a_desc0 = ptx::make_smem_desc(slab_base, 16, 1280, ptx::kLayoutSw128);
    const uint64_t b_desc0 = ptx::make_smem_desc(bring_base, 16, 1024, ptx::kLayoutSw128);
    uint32_t it = 0, sb = 0, bph = 0;
    SlabCursor<NS> q;
    bool ok = true;
    int ti = 0;
    if (ptx::elect_one()) {   // ONE lane runs the whole issue loop: no per-stage elect / warp reconvergence between MMAs
    for (int id = first_tile; id < p.halo_total_tiles && ok && leader; id += tile_step, ++it) {
      const uint32_t as = it & 1;
      if (tr) trace_ev(p, 0, ti, 1);
      ok = ptx::mbar_wait(bar.tmem_empty(as), ((it >> 1) & 1) ^ 1, p.dbg, 13);
      if (!ok) break;
      if (tr) trace_ev(p, 0, ti, 2);
      ptx::tc_fence_after();
      const uint32_t acc = tmem_base + as * kAccCols;
      for (int j = 0; j < nch && ok; ++j) {
        // a ragged last chunk (C_in = 32: half of the 64-channel chunk is TMA zero fill) issues only the K=16 steps that
        // hold real channels
        const int ks = j == p.nch0 - 1 ? p.ksteps0_last : (j == nch - 1 && p.nch1 > 0 ? p.ksteps1_last : 4);
#pragma unroll 1
        for (int kd = 0; kd < 3 && ok; ++kd) {
          uint32_t ph;
          if (kd == 0) {
            for (int pl = 0; pl < TD && ok; ++pl) { const uint32_t sl = q.slot(pl, ph); ok = ptx::mbar_wait(bar.slab_full(sl), ph, p.dbg, 14); }
          } else {
            const uint32_t sl = q.slot(kd + TD - 1, ph);
            ok = ptx::mbar_wait(bar.slab_full(sl), ph, p.dbg, 14);
          }
          if (!ok) break;
          if (tr) trace_ev(p, 0, ti, 3);
          uint64_t a_pl[TD];
#pragma unroll
          for (int pl = 0; pl < TD; ++pl) a_pl[pl] = a_desc0 + (uint64_t)(q.slot(pl + kd, ph) * (uint32_t)(kSlabBytes >> 4));
          const uint32_t first_kd = (j | kd) != 0 ? 1u : 0u;
          // slab released by this kd step: slab kd (last used at kd = min(index, 2)); after kd = 2 also slabs 3 .. TD+1
          const uint32_t rel0 = q.slot(kd, ph), rel1 = TD == 2 ? q.slot(3, ph) : 0u;
#pragma unroll 1
          for (int kh = 0; kh < 3 && ok; ++kh) {
#pragma unroll
            for (int g = 0; g < 3 / TPS; ++g) {   // TPS=3: one stage per kh row; TPS=1: three stages
              ok = ptx::mbar_wait(bar.b_full(sb), bph, p.dbg, 15);
              if (!ok) break;
              ptx::tc_fence_after();
              {
                const uint64_t db0 = b_desc0 + (uint64_t)(sb * (kBBytes >> 4));
#pragma unroll
                for (int u = 0; u < TPS; ++u) {
                  const int kw = TPS == 3 ? u : g;
                  const uint32_t first = (kw != 0) ? 1u : (first_kd | (kh != 0 ? 1u : 0u));
#pragma unroll
                  for (int pl = 0; pl < TD; ++pl) {
                    if (pl < pl_lo || pl >= pl_hi) continue;
                    const uint64_t da = a_pl[pl] + (uint64_t)(kh * kKhUnits + kw * 8);   // (kh*10+kw) rows of 128 B in 16-B units
                    const uint64_t db = db0 + (uint64_t)(u * (kTapBytes >> 4));
                    mma(acc + pl * BLOCK_N, da, db, first);
                    if (ks > 1) mma(acc + pl * BLOCK_N, da + 2, db + 2, 1u);
                    if (ks > 2) mma(acc + pl * BLOCK_N, da + 4, db + 4, 1u);
                    if (ks > 3) mma(acc + pl * BLOCK_N, da + 6, db + 6, 1u);
                  }
                }
                commit(bar.b_empty(sb));
                if (kh == 2 && g == 3 / TPS - 1) {   // last stage of this kd step: release its slab(s) in the same breath
                  commit(bar.slab_empty(rel0));
                  if (kd == 2 && TD == 2) commit(bar.slab_empty(rel1));
                }
              }
              if (++sb == NB) { sb = 0; bph ^= 1; }
            }
          }
          if (!ok) break;
          if (tr) trace_ev(p, 0, ti, 4);
        }
        q.advance(TD + 2);
      }
      // shortcut: TPS chunks per weight stage, each one tap (the slab's centre) on its own TD slabs, released chunk by chunk
      for (int j0 = 0; j0 < sc_nch && ok; j0 += TPS) {
        ok = ptx::mbar_wait(bar.b_full(sb), bph, p.dbg, 15);
        if (!ok) break;
        const uint64_t db0 = b_desc0 + (uint64_t)(sb * (kBBytes >> 4));
#pragma unroll 1
        for (int u = 0; u < TPS && j0 + u < sc_nch && ok; ++u) {
          const int j = j0 + u;
          const int ks = j == p.sc_nch0 - 1 ? p.sc_ksteps0_last : (j == sc_nch - 1 && p.sc_nch1 > 0 ? p.sc_ksteps1_last : 4);
          uint32_t ph;
          for (int pl = 0; pl < TD && ok; ++pl) { const uint32_t sl = q.slot(pl, ph); ok = ptx::mbar_wait(bar.slab_full(sl), ph, p.dbg, 14); }
          if (!ok) break;
          ptx::tc_fence_after();
#pragma unroll
          for (int pl = 0; pl < TD; ++pl) {
            if (pl < pl_lo || pl >= pl_hi) continue;
            const uint64_t da = a_desc0 + (uint64_t)(q.slot(pl, ph) * (uint32_t)(kSlabBytes >> 4)) + (uint64_t)(kKhUnits + 8);   // kh = kw = 1
            const uint64_t db = db0 + (uint64_t)(u * (kTapBytes >> 4));
            mma(acc + pl * BLOCK_N, da, db, 1u);
            if (ks > 1) mma(acc + pl * BLOCK_N, da + 2, db + 2, 1u);
            if (ks > 2) mma(acc + pl * BLOCK_N, da + 4, db + 4, 1u);
            if (ks > 3) mma(acc + pl * BLOCK_N, da + 6, db + 6, 1u);
          }
#pragma unroll
          for (int pl = 0; pl < TD; ++pl) commit(bar.slab_empty(q.slot(pl, ph)));
          q.advance(TD);
        }
        commit(bar.b_empty(sb));
        if (++sb == NB) { sb = 0; bph ^= 1; }
      }
      commit(bar.tmem_full(as));
    }
    }   // elected lane
    __syncwarp();
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue: 8 warps; TMEM lane quarter = warp % 4, column half = (warp - 4) / 4 =====================
    // Measured on B200 (64->64 @ 32^3): with 4 warps the epilogue of a tile took as long as the tile's MMA phase and any
    // extra work (residual read, SiLU) made the kernel epilogue-bound; two warps per lane quarter split the columns, and
    // the residual is fetched into registers BEFORE the accumulator is ready.
    constexpr int kHalfCols = BLOCK_N >= 32 ? BLOCK_N / 2 : BLOCK_N;
    constexpr int kChunks = kHalfCols / 16;
    const int qd = warp & 3;
    const int half = (warp - 4) >> 2;
    const bool active = BLOCK_N >= 32 || half == 0;
    const int cbase = BLOCK_N >= 32 ? half * kHalfCols : 0;
    const int r = qd * 32 + lane;
    const int iw = r & 7, ih = PAIR ? (r >> 4) : (r >> 3), idp = PAIR ? ((r >> 3) & 1) : 0;   // PAIR: row group = h * 2 + d
    const int64_t vox_per = (int64_t)p.out_d * p.out_h * p.out_w;
    uint32_t it = 0;
    int ti = 0;
    uint32_t nstore = 0;   // staged epilogue: plane stores issued so far (selects the staging buffer)
    // fused update: the step's coefficients, Philox key and sample base (uniform over the launch)
    upd::Coef uk = {};
    uint64_t useed = 0;
    int64_t usid0 = 0;
    bool ugen = false;
    uint32_t xround = 0;   // rounds so far: parity of the x_t barrier
    if constexpr (FUSE_UPD) {
      uk = upd::load_coef(p.upd);
      useed = p.upd.seed; usid0 = p.upd.sample_id0;
      if ((p.upd.reserved & 1) && p.upd.t_dev) {
        useed = (uint64_t)(uint32_t)p.upd.t_dev[4] | ((uint64_t)(uint32_t)p.upd.t_dev[5] << 32);
        usid0 += (int64_t)((uint64_t)(uint32_t)p.upd.t_dev[6] | ((uint64_t)(uint32_t)p.upd.t_dev[7] << 32));
      }
      ugen = p.upd.sampler == 0 && uk.t > 0;
    }
    for (int id = first_tile; id < p.halo_total_tiles; id += tile_step, ++it) {
      if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 18);
      const Tile t = decode_tile<PAIR>(p, id);
      const uint32_t as = it & 1;
      const int ow = t.w0 + iw, oh = t.h0 + ih;
      const int colt = t.n_tile * BLOCK_N + cbase;       // first output channel of this warp
      if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 19);
      // residual rows of this thread -> registers while the MMAs of this tile are still running
      bf16x8 rpre[TD][kChunks][2];
      const bool pre = !FUSE_UPD && p.residual != nullptr && active && colt + kHalfCols <= p.c_out;
      if (pre) {
#pragma unroll
        for (int pl = 0; pl < TD; ++pl) {
          const int od = t.d0 + pl + idp;
          if (ow < p.out_w && oh < p.out_h && od < p.out_d) {
            const int64_t vox = ((int64_t)od * p.out_h + oh) * p.out_w + ow;
            const bf16x8* rp = reinterpret_cast<const bf16x8*>(p.residual + ((int64_t)t.n * vox_per + vox) * p.c_out + colt);
#pragma unroll
            for (int c = 0; c < kChunks; ++c) { rpre[pl][c][0] = ldg_bf16x8(rp + 2 * c); rpre[pl][c][1] = ldg_bf16x8(rp + 2 * c + 1); }
          }
        }
      }
      // bias + temb row of this tile's sample -> smem once per tile (double-buffered by accumulator stage)
      float* bs = bias_s + as * 2 * BLOCK_N;
      float* scs = bs + BLOCK_N;
      const bool has_bs = p.bias != nullptr || p.chan_bias != nullptr || p.out_scale != nullptr;
      const bool has_sc = p.out_scale != nullptr;
      if (has_bs) stage_tile_bias<BLOCK_N>(p, bs, scs, t.n, t.n_tile * BLOCK_N, &ti);
      if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 10);
      const bool ok = ptx::mbar_wait(bar.tmem_full(as), (it >> 1) & 1, p.dbg, 16);
      ptx::tc_fence_after();
      if (!ok) break;
      if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 11);
      if constexpr (FUSE_UPD) {
        // eps tile -> x_{t-1}: rounds of 32 columns per thread (one 128-byte line of x_t, fetched one round ahead into
        // registers), fp32 result + 16-bit copy staged in shared memory, two TMA stores per column half and round
        // Rounds of 16 columns per thread; the staging is two SETS of tiles (per column half: 128 rows x 16 fp32 = 8 KB and
        // x 16 bit = 4 KB), used alternately: round q writes set q & 1 while the TMA stores of round q - 1 still read the other
        // one, so no round waits for its predecessor's stores (with one set of 32-column tiles that wait was 2.5 k of a
        // 7.6 k-cycle round).
        constexpr int kRounds = kHalfCols / 16, kQ = TD * kRounds;
        const uint32_t sample = (uint32_t)(usid0 + t.n);
        bool xok = true;
        // (not unrolled: one round is ~1 k instructions -- Philox, Box-Muller, the posterior -- and eight copies of it would
        // not fit the instruction cache next to the issuer / producer loops)
#pragma unroll 1
        for (int q = 0; q < kQ && xok; ++q, ++xround) {
          const int pl = q / kRounds, rd = q % kRounds;
          const int od = t.d0 + pl;
          if (od >= p.out_d) break;   // CTA-uniform
          const uint32_t set = xround & 1;
          uint8_t* stg = stg_base + set * 16384 + half * 8192;
          uint8_t* stg16 = stg16_base + set * 8192 + half * 4096;
          const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + as * kAccCols + pl * BLOCK_N + cbase;
          // All TMA traffic of the round -- the x_t tiles in, x_{t-1} fp32 + 16-bit out -- is issued by the agent warp (warp 12,
          // below): these threads only wait for the x_t tile (x_bar), and signal their writes (w_bar) without waiting for anyone.
          if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 13);
          uint32_t ra[16];
          ptx::tc_ld_32x32b_x16(taddr + rd * 16, ra);
          ptx::tc_wait_ld();
          const int64_t vox = ((int64_t)od * p.out_h + oh) * p.out_w + ow;
          const uint32_t ctr0 = (uint32_t)((vox * p.c_out + colt + rd * 16) >> 2);   // Philox counter = element / 4 of the sample
          xok = upd_epilogue16(p, ra, r, has_bs ? bs + cbase + rd * 16 : nullptr, has_sc ? scs + cbase + rd * 16 : nullptr, uk, ugen, ctr0,
                               sample, useed, stg, stg16, x_bar(set), (xround >> 1) & 1);
          if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 14);
          ptx::fence_proxy_async();      // this thread's tile writes -> visible to the TMA unit
          ptx::tc_fence_before();        // ... and its TMEM reads ordered before the arrival (the agent releases the stage on it)
          ptx::mbar_arrive(w_bar(set));
        }
        if (!xok) break;
        nstore = 0;
      } else if (STAGED && p.y_f32) {
        // fp32 output (eps of the U-Net): 32-column groups of 128-byte rows; the staging area (two 16 KB slots) holds one
        // group per column half, so BLOCK_N = 128 takes two rounds per plane
        constexpr int kRounds = kHalfCols / 32;
#pragma unroll
        for (int pl = 0; pl < TD; ++pl) {
          const int od = t.d0 + pl;
          if (od >= p.out_d) break;   // CTA-uniform
          uint8_t* stg = stg_base + half * 16384;
          const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + as * kAccCols + pl * BLOCK_N + cbase;
#pragma unroll
          for (int rd = 0; rd < kRounds; ++rd) {
            if (warp == 4 && lane == 0) ptx::bulk_wait_read_all();   // the previous round's stores have left the staging
            epilogue_bar_sync256();
            uint32_t ra[16], rb[16];
            ptx::tc_ld_32x32b_x16(taddr + rd * 32, ra);
            ptx::tc_ld_32x32b_x16(taddr + rd * 32 + 16, rb);
            ptx::tc_wait_ld();
            conv_epilogue16_staged_f32(p, ra, r, 0, has_bs ? bs + cbase + rd * 32 : nullptr, has_sc ? scs + cbase + rd * 32 : nullptr,
                                       stg, pre, rpre[pl][2 * rd]);
            conv_epilogue16_staged_f32(p, rb, r, 16, has_bs ? bs + cbase + rd * 32 + 16 : nullptr,
                                       has_sc ? scs + cbase + rd * 32 + 16 : nullptr, stg, pre, rpre[pl][2 * rd + 1]);
            ptx::fence_proxy_async();
            epilogue_bar_sync256();
            if (warp == 4 && lane == 0) {
              for (int h = 0; h < 2; ++h) {
                const int col = t.n_tile * BLOCK_N + h * kHalfCols + rd * 32;
                if (col < p.c_out) ptx::tma_store_5d(&mapY, ptx::smem_u32(stg_base + h * 16384), col, t.w0, t.h0, od, t.n);
              }
              ptx::bulk_commit_group();
            }
          }
        }
        nstore = 0;   // (buffer rotation is a bf16-path notion)
      } else if constexpr (STAGED) {
#pragma unroll
        for (int pl = 0; pl < TD; ++pl) {
          const int od = t.d0 + pl;
          if (od >= p.out_d) break;   // CTA-uniform
          const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + as * kAccCols + pl * BLOCK_N + cbase;
          store_plane16<BLOCK_N, PAIR>(p, &mapY, stg_base, nstore, taddr, r, cbase, t.n_tile * BLOCK_N, bs, scs, has_bs, has_sc,
                                       t.w0, t.h0, od, t.n, pre, rpre[pl], &ti);
          ++nstore;
        }
      } else
      if (active) {
#pragma unroll
        for (int pl = 0; pl < TD; ++pl) {
          const int od = t.d0 + pl;
          const bool valid = ow < p.out_w && oh < p.out_h && od < p.out_d;
          const int64_t vox = ((int64_t)od * p.out_h + oh) * p.out_w + ow;
          const int64_t row_off = ((int64_t)t.n * vox_per + vox) * p.c_out;
          const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + as * kAccCols + pl * BLOCK_N + cbase;
#pragma unroll
          for (int c = 0; c < kChunks; c += 2) {
            const int col0 = colt + c * 16;
            if (col0 >= p.c_out) break;
            uint32_t ra[16], rb[16];
            ptx::tc_ld_32x32b_x16(taddr + c * 16, ra);
            if (c + 1 < kChunks) ptx::tc_ld_32x32b_x16(taddr + c * 16 + 16, rb);
            ptx::tc_wait_ld();
            if (valid) {
              conv_epilogue16(p, ra, col0, t.n, vox, vox_per, row_off, has_bs ? bs + cbase + c * 16 : nullptr, nullptr,
                              has_sc ? scs + cbase + c * 16 : nullptr, pre ? rpre[pl][c] : nullptr);
              if (c + 1 < kChunks && col0 + 16 < p.c_out)
                conv_epilogue16(p, rb, col0 + 16, t.n, vox, vox_per, row_off, has_bs ? bs + cbase + c * 16 + 16 : nullptr, nullptr,
                                has_sc ? scs + cbase + c * 16 + 16 : nullptr, pre ? rpre[pl][c + 1 < kChunks ? c + 1 : c] : nullptr);
            }
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (warp == 4 && lane == 0) trace_ev(p, 1, ti, 12);
      // (FUSE_UPD: the agent warp releases the accumulator stage once the tile's last round is complete -- the cluster-scope
      // arrive costs the arriving warp ~2.5 k cycles, which these warps would pay at every tile boundary)
      if (!FUSE_UPD) release_acc<CG2>(p, bar.tmem_empty(as), id, tile_step);
    }
    if (STAGED && !FUSE_UPD && warp == 4 && lane == 0) ptx::bulk_wait_read_all();   // smem must outlive the last store's reads
  }
  if constexpr (FUSE_UPD) {
    if (warp == 12 && lane < 4) {
      // ===================== TMA agent of the fused update (4 lanes, each with its own bulk-group bookkeeping) =====================
      // lane 0 / 2: the fp32 tile of column half 0 / 1 (x_t load, x_{t-1} store); lane 1 / 3: its 16-bit tile (store).  Per round:
      // wait until the 256 epilogue threads have written the tiles of set r & 1 (w_bar), store them, wait until that store has
      // read its tile, and request the x_t tiles of round r + 2 into the same set (x_bar[set]: 2 loads + 2 plain arrivals) -- a
      // whole round before they are needed.  With the TMA instructions on epilogue lanes every round paid ~750 cycles of issue
      // latency inside the warps that do the arithmetic, and the x_t tile of a round was requested only at its start.
      constexpr int kHalfColsA = BLOCK_N / 2, kRoundsA = kHalfColsA / 16;
      const int h = lane >> 1;
      const bool f32 = (lane & 1) == 0;
      auto rounds_of = [&](const Tile& t) { const int pls = p.out_d - t.d0 < TD ? p.out_d - t.d0 : TD; return pls * kRoundsA; };
      auto request_x = [&](const Tile& t, int q, uint32_t rnd) {
        if (f32) {
          ptx::mbar_expect_tx(x_bar(rnd & 1), 8192u);
          ptx::tma_load_5d(ptx::smem_u32(stg_base + (rnd & 1) * 16384 + h * 8192), &mapY, x_bar(rnd & 1),
                           t.n_tile * BLOCK_N + h * kHalfColsA + (q % kRoundsA) * 16, t.w0, t.h0, t.d0 + q / kRoundsA, t.n);
        } else {
          ptx::mbar_arrive(x_bar(rnd & 1));
        }
      };
      // look-ahead cursor: (tile id, round within the tile) of round `rnd + 2`
      int id2 = first_tile, q2 = 0;
      Tile t2 = decode_tile<PAIR>(p, id2 < p.halo_total_tiles ? id2 : 0);
      auto advance2 = [&]() {
        if (++q2 >= rounds_of(t2)) { q2 = 0; id2 += tile_step; if (id2 < p.halo_total_tiles) t2 = decode_tile<PAIR>(p, id2); }
      };
      for (uint32_t r0 = 0; r0 < 2 && id2 < p.halo_total_tiles; ++r0) { request_x(t2, q2, r0); advance2(); }   // both sets are free at the start
      uint32_t rnd = 0, atile = 0;   // rounds / tiles so far
      bool ok = true;
      for (int id = first_tile; id < p.halo_total_tiles && ok; id += tile_step) {
        const Tile t = decode_tile<PAIR>(p, id);
        const int nq = rounds_of(t);
        for (int q = 0; q < nq; ++q, ++rnd) {
          ok = ptx::mbar_wait(w_bar(rnd & 1), (rnd >> 1) & 1, p.dbg, 18);
          if (!ok) break;
          const int col = t.n_tile * BLOCK_N + h * kHalfColsA + (q % kRoundsA) * 16, od = t.d0 + q / kRoundsA;
          if (f32) ptx::tma_store_5d(&mapY, ptx::smem_u32(stg_base + (rnd & 1) * 16384 + h * 8192), col, t.w0, t.h0, od, t.n);
          else ptx::tma_store_5d(&mapZ, ptx::smem_u32(stg16_base + (rnd & 1) * 8192 + h * 4096), col, t.w0, t.h0, od, t.n);
          ptx::bulk_commit_group();
          if (id2 < p.halo_total_tiles) {
            ptx::bulk_wait_read_all();   // this lane's store has read its tile: the set may be refilled
            request_x(t2, q2, rnd + 2);
            advance2();
          }
          if (q == nq - 1 && lane == 1 && id + 2 * tile_step < p.halo_total_tiles) {   // (nobody waits for the last two tiles' release)
            // the tile's last round is complete: every epilogue thread has read its accumulators (tcgen05.ld -> fence -> w_bar):
            // hand the TMEM stage back to the (leader's) MMA issuers
            ptx::tc_fence_after();
            ptx::tc_fence_before();
            if (CG2) ptx::mbar_arrive_cluster(ptx::mapa_shared(bar.tmem_empty(atile & 1), 0)); else ptx::mbar_arrive(bar.tmem_empty(atile & 1));
          }
        }
        ++atile;
      }
      ptx::bulk_wait_read_all();   // smem must outlive the last stores' reads
    }
    if (warp == 12) __syncwarp();   // the agent's four lanes rejoin their warp before the block-wide barrier
  }
  teardown<CG2>(&p, tmem_base, kTmemCols);
}

}  // namespace halo
