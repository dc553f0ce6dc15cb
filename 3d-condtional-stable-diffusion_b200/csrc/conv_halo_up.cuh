// x2 up-convolutions on the halo-reuse / CTA-pair machinery: nearest-upsample(2) + Conv3 (UpSample, dm3d.py:269-277) and
// Conv3DTranspose(k4, s2) (vqvae3d_monai.py:372-381, vqgan_attn_cp.py:404-412), both re-indexed on the host to 8 output-parity
// sub-convolutions of 2^3 taps on the LOW-resolution input (conv.cu: b200dm_conv_pack_weights).
//
//   tile        8 w x 16 h x 2 d low-resolution voxels, one output parity (pd, ph, pw), BLOCK_N output channels; the tile list
//               enumerates n-tile, spatial pair, parity, half-of-pair: the two CTAs of a pair always share parity and weights
//   slabs       the same 10 x 18 x 64ch halo slabs as conv_halo_kernel; a parity needs input planes d0-1+pd .. d0+1+pd (3 slabs
//               per channel chunk) and reads tap (td, th, tw) at slab offset (th + ph, tw + pw)
//   weights     one stage = the 4 in-plane taps of one td: box {64, BLOCK_N / 2, 4} of the packed [parity][n][chunk*8 + tap] image
//               (each CTA of the pair stages half of the rows)
//   MMA         cta_group::2, M = 256: one issuer warp per output plane in the leader CTA
//   epilogue    staged bf16 tile -> TMA store through the parity's strided output map (ConvOutMaps::y[parity])
//
// The per-tap GEMM kernel ran these layers at 77 us (16^3 -> 32^3, 128 -> 128, B = 8): every tap re-fetched its A tile.
#pragma once
#include "conv_halo.cuh"

namespace halo {

// PAIR: 8 x 8 low-resolution planes (8^3 -> 16^3): the tile is 8 w x 8 h x 2 d from pair slabs (box {64, 10, 2, 10, 1} of a tensor map
// whose dims are listed (C, W, D, H, N), rows [h][d][w] as in conv_halo_kernel's PAIR variant): one accumulator, one issuer warp,
// two pair slabs per channel chunk (td = 0, 1), tap offset (th + ph) * 20 + (tw + pw) rows.
// Shared memory: conv_halo_kernel's layout with 4-tap weight stages of half the rows and the staged epilogue.
template <int BLOCK_N, int NS, int NB, bool PAIR>
using UpSmem = Smem<BLOCK_N, NS, NB, 4, true, PAIR, true, false>;

template <int BLOCK_N, int NS, int NB, bool PAIR = false>
__global__ void __launch_bounds__(kThreads, 1)
conv_halo_up_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                    const __grid_constant__ CUtensorMap mapB, const __grid_constant__ ConvOutMaps om, const ConvParams p) {
  static_assert(BLOCK_N == 32 || BLOCK_N == 64 || BLOCK_N == 128, "32-, 64- or 128-channel tiles");
  constexpr int TD = PAIR ? 1 : 2;                 // accumulators (PAIR: one M = 128 tile spanning two planes)
  constexpr int kSlabsPerChunk = PAIR ? 2 : 3;
  constexpr int kIss = PAIR ? 1 : 2;               // issuer warps
  constexpr int kKhUnits = PAIR ? 160 : 80;
  using L = UpSmem<BLOCK_N, NS, NB, PAIR>;
  constexpr int kSlabBytes = L::kSlabBytes, kSlabTx = PAIR ? 200 * 128 : halo::kSlabTx;
  constexpr int kBRows = L::kBRows;
  constexpr int kTapBytes = L::kTapBytes;
  constexpr int kBBytes = L::kBBytes;
  constexpr uint32_t kAccCols = TD * BLOCK_N;
  constexpr uint32_t kTmemCols = 2 * kAccCols;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* b_ring = smem + L::kBRing;
  uint8_t* stg_base = smem + L::kStage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + L::kTmemPtr);
  float* bias_s = reinterpret_cast<float*>(smem + L::kBias);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t slab_base = ptx::smem_u32(smem);
  const uint32_t bring_base = ptx::smem_u32(b_ring);
  const uint32_t bar_base = ptx::smem_u32(bars);
  const Bars<NS, NB> bar{bar_base};

  pdl_launch_dependents();
  const int nch = p.nch0 + p.nch1;
  const int first_tile = blockIdx.x, tile_step = gridDim.x;
  const uint32_t crank = ptx::cluster_ctarank();
  const bool leader = crank == 0;

  // tile id -> (parity, n-tile, sample, d0, h0, w0); ids 2k, 2k+1 differ only in the spatial position
  struct UTile { int w0, h0, d0, n, nt, par; };
  auto decode = [&](int id) {
    UTile t;
    // n-tile outermost, then the spatial pair, then the 8 parities, then the half of the pair: the 8 parities of one
    // position read the same input slabs back to back (parity outermost re-read the input from DRAM: 4.3 GB for a 1.1 GB
    // tensor at 64^3 x 64, L2 hit rate 32 %)
    const int per8 = p.halo_tiles_per_ntile * 8;
    t.nt = id / per8;
    const int rem = id - t.nt * per8;
    t.par = (rem >> 1) & 7;
    int r = ((rem >> 4) << 1) | (rem & 1);
    t.w0 = (r % p.tiles_w) * 8; r /= p.tiles_w;
    t.h0 = (r % p.tiles_h) * (PAIR ? 8 : 16); r /= p.tiles_h;
    t.d0 = (r % p.tiles_d) * 2; r /= p.tiles_d;
    t.n = r;
    return t;
  };

  if (threadIdx.x == 0) {
    bar.init(kIss, 16);
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&mapA0);
    ptx::prefetch_tmap(&mapB);
  }
  if (warp == 2) tmem_alloc<true>(tmem_ptr_smem, kTmemCols);
  const uint32_t tmem_base = setup_join<true>(tmem_ptr_smem);

  if (warp == 0) {
    // ===================== slab producer: 3 slabs per channel chunk =====================
    uint32_t s = 0, ph = 1;
    bool ok = true;
    for (int id = first_tile; id < p.halo_total_tiles && ok; id += tile_step) {
      const UTile t = decode(id);
      const int pd = (t.par >> 2) & 1;
      for (int j = 0; j < nch && ok; ++j) {
        const CUtensorMap* map = j < p.nch0 ? &mapA0 : &mapA1;
        const int c0 = (j < p.nch0 ? j : j - p.nch0) * 64;
        for (int pl = 0; pl < kSlabsPerChunk; ++pl) {
          ok = ptx::mbar_wait(bar.slab_empty(s), ph, p.dbg, 41);
          if (!ok) break;
          if (ptx::elect_one()) {
            if (leader) ptx::mbar_expect_tx(bar.slab_full(s), 2 * kSlabTx);
            if (PAIR) ptx::tma_load_5d_cg2(slab_base + s * kSlabBytes, map, ptx::mapa_shared(bar.slab_full(s), 0), c0, t.w0 - 1,
                                           t.d0 - 1 + pd + pl, t.h0 - 1, t.n);
            else ptx::tma_load_5d_cg2(slab_base + s * kSlabBytes, map, ptx::mapa_shared(bar.slab_full(s), 0), c0, t.w0 - 1, t.h0 - 1,
                                      t.d0 - 1 + pd + pl, t.n);
          }
          __syncwarp();
          if (++s == NS) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== weight producer: one stage per (chunk, td) = 4 in-plane taps =====================
    produce_weights<NS, NB, kBRows, kBBytes, true>(p, bar, &mapB, bring_base, crank, first_tile, tile_step, nch * 2, 4, 42, [&](int id) {
      const UTile t = decode(id);
      return t.par * p.n_pad + t.nt * BLOCK_N;
    });
  } else if (warp == 2 || (warp == 3 && kIss == 2)) {
    // ===================== MMA issuers (leader CTA): warp 2 -> output plane 0, warp 3 -> plane 1 =====================
    const int pl = warp - 2;
    constexpr uint32_t idesc = ptx::make_idesc_act(256, BLOCK_N);
    const uint64_t a_desc0 = ptx::make_smem_desc(slab_base, 16, 1280, ptx::kLayoutSw128);
    const uint64_t b_desc0 = ptx::make_smem_desc(bring_base, 16, 1024, ptx::kLayoutSw128);
    if (leader && ptx::elect_one()) {
      uint32_t it = 0, sb = 0, bph = 0;
      SlabCursor<NS> q;
      bool ok = true;
      for (int id = first_tile; id < p.halo_total_tiles && ok; id += tile_step, ++it) {
        const UTile t = decode(id);
        const int ph_ = (t.par >> 1) & 1, pw_ = t.par & 1;
        const uint32_t as = it & 1;
        ok = ptx::mbar_wait(bar.tmem_empty(as), ((it >> 1) & 1) ^ 1, p.dbg, 43);
        if (!ok) break;
        ptx::tc_fence_after();
        const uint32_t acc = tmem_base + as * kAccCols + pl * BLOCK_N;
        for (int j = 0; j < nch && ok; ++j) {
          const int ks = j == p.nch0 - 1 ? p.ksteps0_last : (j == nch - 1 && p.nch1 > 0 ? p.ksteps1_last : 4);
#pragma unroll 1
          for (int td = 0; td < 2 && ok; ++td) {
            uint32_t phs;
            if (PAIR) {   // pair slab td
              const uint32_t sl = q.slot(td, phs);
              ok = ptx::mbar_wait(bar.slab_full(sl), phs, p.dbg, 44);
            } else if (td == 0) {
              for (int i = 0; i < TD && ok; ++i) { const uint32_t sl = q.slot(i, phs); ok = ptx::mbar_wait(bar.slab_full(sl), phs, p.dbg, 44); }
            } else {
              const uint32_t sl = q.slot(TD, phs);
              ok = ptx::mbar_wait(bar.slab_full(sl), phs, p.dbg, 44);
            }
            if (!ok) break;
            const uint64_t a_pl = a_desc0 + (uint64_t)(q.slot(pl + td, phs) * (uint32_t)(kSlabBytes >> 4));
            ok = ptx::mbar_wait(bar.b_full(sb), bph, p.dbg, 45);
            if (!ok) break;
            ptx::tc_fence_after();
            const uint64_t db0 = b_desc0 + (uint64_t)(sb * (kBBytes >> 4));
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const uint64_t da = a_pl + (uint64_t)((((u >> 1) + ph_) * kKhUnits) + ((u & 1) + pw_) * 8);
              const uint64_t db = db0 + (uint64_t)(u * (kTapBytes >> 4));
              ptx::tc_mma_f16_cg2(acc, da, db, idesc, (j | td | u) != 0 ? 1u : 0u);
              if (ks > 1) ptx::tc_mma_f16_cg2(acc, da + 2, db + 2, idesc, 1u);
              if (ks > 2) ptx::tc_mma_f16_cg2(acc, da + 4, db + 4, idesc, 1u);
              if (ks > 3) ptx::tc_mma_f16_cg2(acc, da + 6, db + 6, idesc, 1u);
            }
            ptx::tc_commit_cg2(bar.b_empty(sb), (uint16_t)3);
            if (PAIR) {
              ptx::tc_commit_cg2(bar.slab_empty(q.slot(td, phs)), (uint16_t)3);
            } else if (td == 0) {
              ptx::tc_commit_cg2(bar.slab_empty(q.slot(0, phs)), (uint16_t)3);
            } else {
              ptx::tc_commit_cg2(bar.slab_empty(q.slot(1, phs)), (uint16_t)3);
              ptx::tc_commit_cg2(bar.slab_empty(q.slot(2, phs)), (uint16_t)3);
            }
            if (++sb == NB) { sb = 0; bph ^= 1; }
          }
          q.advance(kSlabsPerChunk);
        }
        ptx::tc_commit_cg2(bar.tmem_full(as), (uint16_t)3);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== epilogue: 8 warps; lane quarter = warp % 4, column half = (warp - 4) / 4 =====================
    const int qd = warp & 3;
    const int cbase = ((warp - 4) >> 2) * (BLOCK_N / 2);   // column half
    const int r = qd * 32 + lane;
    uint32_t it = 0, nstore = 0;
    for (int id = first_tile; id < p.halo_total_tiles; id += tile_step, ++it) {
      const UTile t = decode(id);
      const uint32_t as = it & 1;
      float* bs = bias_s + as * 2 * BLOCK_N;
      float* scs = bs + BLOCK_N;
      const bool has_bs = p.bias != nullptr || p.chan_bias != nullptr || p.out_scale != nullptr;
      const bool has_sc = p.out_scale != nullptr;
      if (has_bs) stage_tile_bias<BLOCK_N>(p, bs, scs, t.n, t.nt * BLOCK_N, nullptr);
      const bool ok = ptx::mbar_wait(bar.tmem_full(as), (it >> 1) & 1, p.dbg, 46);
      ptx::tc_fence_after();
      if (!ok) break;
#pragma unroll
      for (int pl = 0; pl < TD; ++pl) {
        const int od = t.d0 + pl;            // low-resolution (M-space) plane; the parity map places it at 2 * od + pd
        if (od >= p.m_d) break;              // CTA-uniform
        const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + as * kAccCols + pl * BLOCK_N + cbase;
        store_plane16<BLOCK_N, PAIR>(p, &om.y[t.par], stg_base, nstore, taddr, r, cbase, t.nt * BLOCK_N, bs, scs, has_bs, has_sc,
                                     t.w0, t.h0, od, t.n, false, nullptr, nullptr);
        ++nstore;
      }
      ptx::tc_fence_before();
      __syncwarp();
      release_acc<true>(p, bar.tmem_empty(as), id, tile_step);
    }
    if (warp == 4 && lane == 0) ptx::bulk_wait_read_all();
  }
  teardown<true>(nullptr, tmem_base, kTmemCols);
}

}  // namespace halo
