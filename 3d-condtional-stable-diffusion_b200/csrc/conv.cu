// K1-K5 (+ the attention matmuls): Conv3D as an implicit GEMM on the 5th-gen tensor cores.
//
//   GEMM view   M = output voxels (tile = a 128-voxel box bw x bh x bd x bn of the NDHWC tensor)
//               N = C_out (BLOCK_N columns of TMEM, fp32 accumulators)
//               K = taps x C_in, walked as k-blocks of (tap, 64-channel chunk)
//   A operand   TMA (cp.async.bulk.tensor.5d, SWIZZLE_128B) loads the box shifted by the tap offset straight
//               from the bf16 NDHWC activation: out-of-bounds voxels / channels are zero-filled by the TMA
//               unit, which IS TF 'same' padding (incl. the asymmetric (0,1) of stride-2) -- no im2col
//               buffer, no padded copy.  Two K-segments (two tensor maps) read [x, skip] without ever
//               materialising layers.Concatenate.
//   B operand   packed bf16 weights [group][n_pad][chunk][tap][64], one 2-D TMA per k-block.
//   MMA         tcgen05.mma.cta_group::1.kind::f16, M=128, N=BLOCK_N, K=16 x4 per k-block, issued by one
//               thread; accumulators live in TMEM; tcgen05.commit releases smem stages / signals the epilogue.
//   Epilogue    4 warps: tcgen05.ld -> +bias +temb[t][n] -> PReLU/act -> +residual -> act -> bf16|fp32 NDHWC
//               (optionally transposed per sample, for V^T of the attention blocks).
//   PARITY mode nearest-upsample(2)+Conv3 and ConvTranspose(k4,s2) both become 8 output-parity
//               sub-convolutions of 2^3 taps on the low-res input (blockIdx.z = parity): 27 -> 8 taps.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2-5 = epilogue.
#include <cuda.h>
#include <string.h>
#include <math.h>
#include <memory>
#include <new>
#include <utility>
#include "conv_common.cuh"

#include "conv_halo.cuh"
#include "conv_halo_up.cuh"
#include "conv_stencil.cuh"
#include "conv_sweep.cuh"

namespace {

constexpr int kThreads = 192;
constexpr int kABytes = 128 * 128;  // 128 rows x 64 bf16

// Shared-memory layout of conv_igemm_kernel, offsets from the 1024-aligned base: NSTAGE x (A tile | B tile) | staged residual
// tile (plans with a residual and the staged epilogue only) | barriers | TMEM address | bias + scale [2][BLOCK_N].
template <int BLOCK_N, int NSTAGE>
struct GemmSmem {
  static constexpr int kStageBytes = kABytes + BLOCK_N * 128;
  static constexpr int kResBytes = BLOCK_N >= 64 ? BLOCK_N * 256 : 0;   // 128 rows x BLOCK_N bf16 residual tile
  // [0..NSTAGE) full, [NSTAGE..2NSTAGE) empty, [2NSTAGE] tmem_full, [2NSTAGE+1] residual tile (+1 keeps the bias 16-byte aligned)
  static constexpr int kBars = 2 * NSTAGE + 3;
  static constexpr size_t kRes = (size_t)NSTAGE * kStageBytes;
  static constexpr size_t kTmemPtr = kBars * 8;       // from the barriers, as is the bias
  static constexpr size_t kBias = kTmemPtr + 8;
  __host__ __device__ static constexpr size_t bar_off(bool staged_res) { return kRes + (staged_res ? kResBytes : 0); }
  // with the alignment slack; 16 bytes are reserved for the 8-byte TMEM address
  static constexpr size_t bytes(bool staged_res) { return 1024 + bar_off(staged_res) + kTmemPtr + 16 + 2 * BLOCK_N * 4; }
};

// Split-K: adds the partial accumulators of the cluster's other ks - 1 CTAs (staged as fp32 [col / 4][row] float4 in their
// shared memory, read through DSMEM) to NB blocks of 16 accumulator columns c0 + 16 b .. of row r.
template <int NB>
__device__ __forceinline__ void add_peer_partials(uint32_t (&rr)[NB][16], const float* stage_f, int c0, int r, int ks) {
  for (int pr = 1; pr < ks; ++pr) {
    const uint32_t remote = ptx::mapa_shared(ptx::smem_u32(stage_f + c0 * 128 + r * 4), (uint32_t)pr);
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const float4 a4 = ptx::ld_dsmem_f32x4(remote + (16 * b + j) * 512);
        rr[b][j] = __float_as_uint(__uint_as_float(rr[b][j]) + a4.x); rr[b][j + 1] = __float_as_uint(__uint_as_float(rr[b][j + 1]) + a4.y);
        rr[b][j + 2] = __float_as_uint(__uint_as_float(rr[b][j + 2]) + a4.z); rr[b][j + 3] = __float_as_uint(__uint_as_float(rr[b][j + 3]) + a4.w);
      }
    }
  }
}

// KSPLIT: split-K cluster (K range per CTA, partial accumulators reduced through distributed shared memory by the cluster's
// first CTA); four-stage instantiations only.
// (two-stage instantiations: registers capped so that four CTAs share an SM -- see select_variant)
template <int BLOCK_N, int NSTAGE, bool KSPLIT>
__global__ void __launch_bounds__(kThreads, NSTAGE == 2 ? 4 : 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                  const __grid_constant__ CUtensorMap mapB, const __grid_constant__ ConvOutMaps om, const ConvParams p) {
  using L = GemmSmem<BLOCK_N, NSTAGE>;
  constexpr int kStageBytes = L::kStageBytes;
  constexpr uint32_t kTmemCols = BLOCK_N < 32 ? 32 : BLOCK_N;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const bool staged = BLOCK_N >= 64 && p.tma_epi != 0;
  const bool staged_res = staged && p.residual != nullptr;
  uint8_t* res_smem = smem + L::kRes;
  uint8_t* bar_smem = smem + L::bar_off(staged_res);
  uint64_t* bars = reinterpret_cast<uint64_t*>(bar_smem);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bar_smem + L::kTmemPtr);
  float* bias_s = reinterpret_cast<float*>(bar_smem + L::kBias);   // [2][BLOCK_N]: bias (+temb), output-affine scale

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = ptx::smem_u32(smem);
  const uint32_t bar_base = ptx::smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (NSTAGE + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * NSTAGE);
  const uint32_t res_bar = bar_base + 8u * (2 * NSTAGE + 1);

  // tile decode
  pdl_launch_dependents();
  int tix = 0;   // timeline index of this thread's region (tuning aid: b200dm_conv_plan_set_trace)
  if (threadIdx.x == 0) trace_ev(p, 3, tix, 40);
  const int ks = KSPLIT ? p.ksplit : 1;
  const int krank = KSPLIT ? (int)ptx::cluster_ctaid_x() : 0;
  int bx = KSPLIT ? blockIdx.x / ks : blockIdx.x;
  const int tw = bx % p.tiles_w; bx /= p.tiles_w;
  const int th = bx % p.tiles_h; bx /= p.tiles_h;
  const int td = bx % p.tiles_d; bx /= p.tiles_d;
  const int tn = bx;
  const int w0 = tw * p.box_w, h0 = th * p.box_h, d0 = td * p.box_d, n0 = tn * p.box_n;
  const int n_tile = blockIdx.y;
  const int parity = blockIdx.z;
  const int pw = parity & 1, ph = (parity >> 1) & 1, pd = (parity >> 2) & 1;
  const int nkb_all = (p.nch0 + p.nch1) * p.ntaps;
  const int kb0 = KSPLIT ? (int)((long long)krank * nkb_all / ks) : 0;            // this CTA's K range
  const int kb1 = KSPLIT ? (int)((long long)(krank + 1) * nkb_all / ks) : nkb_all;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NSTAGE; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
    ptx::mbar_init(tmem_full_bar, 1);
    ptx::mbar_init(res_bar, 1);
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&mapA0);
    ptx::prefetch_tmap(&mapB);
    if (staged) ptx::prefetch_tmap(&om.y[blockIdx.z]);
  }
  if (warp == 1) {
    ptx::tmem_alloc(ptx::smem_u32(tmem_ptr_smem), kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  bool mid_synced = false;                // split-K: every thread of the cluster passes ONE mid-kernel cluster barrier
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  if (threadIdx.x == 0) trace_ev(p, 3, tix, 41);
  pdl_wait();   // everything above overlapped the previous kernel's tail; from here on we touch its outputs
  if (threadIdx.x == 0) trace_ev(p, 3, tix, 42);

  if (warp == 0) {
    // ===================== TMA producer =====================
    {
      const int b_row = (p.mode == B200DM_CONV_PARITY ? parity : (p.mode == B200DM_CONV_BATCHED_GEMM ? n0 : 0)) * p.n_pad +
                        n_tile * BLOCK_N;
      uint32_t s = 0, phase = 0;
      int chunk = kb0 / p.ntaps, tap = kb0 % p.ntaps;
      if (BLOCK_N >= 64 && staged_res && krank == 0 && ptx::elect_one()) {
        // residual tile (same box as the output tile) -> smem, consumed by the epilogue long after it has landed
        int ng = 0;
        for (int g = 0; g < BLOCK_N / 64; ++g) if (n_tile * BLOCK_N + g * 64 < p.c_out) ++ng;
        ptx::mbar_expect_tx(res_bar, (uint32_t)ng * 16384u);
        for (int g = 0; g < ng; ++g)
          ptx::tma_load_5d(ptx::smem_u32(res_smem) + g * 16384, &om.r, res_bar, n_tile * BLOCK_N + g * 64, w0, h0, d0, n0);
      }
      __syncwarp();
      for (int kb = kb0; kb < kb1; ++kb) {
        if (!ptx::mbar_wait(empty_bar(s), phase ^ 1, p.dbg, 1)) break;
        if (lane == 0 && kb == kb0) trace_ev(p, 3, tix, 43);
        if (ptx::elect_one()) {
          int ow, oh, od;
          if (p.mode == B200DM_CONV_PARITY) {
            ow = (tap & 1) - 1 + pw; oh = ((tap >> 1) & 1) - 1 + ph; od = ((tap >> 2) & 1) - 1 + pd;
          } else {
            const int k = p.ksize;
            ow = tap % k - p.pad; oh = (tap / k) % k - p.pad; od = tap / (k * k) - p.pad;
          }
          const uint32_t a_dst = smem_base + s * kStageBytes;
          const uint32_t b_dst = a_dst + kABytes;
          ptx::mbar_expect_tx(full_bar(s), kStageBytes);
          const CUtensorMap* mapA = chunk < p.nch0 ? &mapA0 : &mapA1;
          const int cch = (chunk < p.nch0 ? chunk : chunk - p.nch0) * 64;
          ptx::tma_load_5d(a_dst, mapA, full_bar(s), cch, w0 * p.stride + ow, h0 * p.stride + oh, d0 * p.stride + od, n0);
          ptx::tma_load_2d(b_dst, &mapB, full_bar(s), kb * 64, b_row);
        }
        __syncwarp();
        if (++s == NSTAGE) { s = 0; phase ^= 1; }
        if (++tap == p.ntaps) { tap = 0; ++chunk; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    {  // whole warp walks the loop; one elected lane issues (no per-lane serialisation loops around UTCHMMA)
      constexpr uint32_t idesc = ptx::make_idesc_act(128, BLOCK_N);
      const uint64_t a_desc0 = ptx::make_smem_desc(smem_base, 16, 1024, ptx::kLayoutSw128);
      const uint64_t b_desc0 = ptx::make_smem_desc(smem_base + kABytes, 16, 1024, ptx::kLayoutSw128);
      bool ok = true;
      uint32_t s = 0, phase = 0;
      int mchunk = kb0 / p.ntaps, mtap = kb0 % p.ntaps;
      for (int kb = kb0; kb < kb1 && ok; ++kb) {
        ok = ptx::mbar_wait(full_bar(s), phase, p.dbg, 2);
        if (!ok) break;
        if (lane == 0) trace_ev(p, 0, tix, 44);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          // swap_ab (BLOCK_N = 128, both tiles [128 rows][64 K]): the weight tile is the A operand -> D^T in TMEM
          const uint64_t da = (p.swap_ab ? b_desc0 : a_desc0) + (uint64_t)(s * (kStageBytes >> 4));
          const uint64_t db = (p.swap_ab ? a_desc0 : b_desc0) + (uint64_t)(s * (kStageBytes >> 4));
          // a ragged last chunk of a K segment (e.g. C_in = 32 or 8) issues only the K=16 steps that hold real channels
          const int ksn = mchunk == p.nch0 - 1 ? p.ksteps0_last : (mchunk == p.nch0 + p.nch1 - 1 && p.nch1 > 0 ? p.ksteps1_last : 4);
          ptx::tc_mma_f16(tmem_base, da, db, idesc, kb != kb0 ? 1u : 0u);
          if (ksn > 1) ptx::tc_mma_f16(tmem_base, da + 2, db + 2, idesc, 1u);
          if (ksn > 2) ptx::tc_mma_f16(tmem_base, da + 4, db + 4, idesc, 1u);
          if (ksn > 3) ptx::tc_mma_f16(tmem_base, da + 6, db + 6, idesc, 1u);
          ptx::tc_commit(empty_bar(s));
        }
        __syncwarp();
        if (++s == NSTAGE) { s = 0; phase ^= 1; }
        if (++mtap == p.ntaps) { mtap = 0; ++mchunk; }
      }
      if (ptx::elect_one()) ptx::tc_commit(tmem_full_bar);
      __syncwarp();
    }
  } else {
    // ===================== epilogue warps (TMEM lane quarter = warp % 4) =====================
    const int q = warp & 3;
    const int r = q * 32 + lane;
    int t = r;
    const int iw = t % p.box_w; t /= p.box_w;
    const int ih = t % p.box_h; t /= p.box_h;
    const int id = t % p.box_d; t /= p.box_d;
    const int in_ = t;
    const int mw = w0 + iw, mh = h0 + ih, md = d0 + id, n = n0 + in_;
    const bool valid = (mw < p.m_w) && (mh < p.m_h) && (md < p.m_d) && (n < p.batch);
    int ow = mw, oh = mh, od = md;
    if (p.mode == B200DM_CONV_PARITY) { ow = 2 * mw + pw; oh = 2 * mh + ph; od = 2 * md + pd; }
    const int64_t vox = ((int64_t)od * p.out_h + oh) * p.out_w + ow;           // voxel index within the sample
    const int64_t vox_per = (int64_t)p.out_d * p.out_h * p.out_w;
    const int64_t row_off = ((int64_t)n * vox_per + vox) * p.c_out;             // NDHWC element offset of channel 0
    // bias (+ temb row when the tile lies inside one sample) -> smem while the MMAs run
    const float* cb = nullptr;
    const float* cbrow = nullptr;
    if (p.chan_bias) {
      const int tt = p.t_dev ? p.t_dev[0] : 0;
      const bool uniform = p.box_n == 1 || p.chan_bias_rows <= 1;
      const float* row = p.chan_bias + ((int64_t)tt * p.chan_bias_rows + (p.chan_bias_rows > 1 ? (uniform ? n0 : n) : 0)) * p.c_out;
      if (uniform) cbrow = n0 < p.batch ? row : nullptr;
      else if (valid) cb = row;
    }
    const bool has_bs = p.bias != nullptr || cbrow != nullptr || p.out_scale != nullptr;
    float* scale_s = bias_s + BLOCK_N;
    if (has_bs) {
      stage_bias(p, bias_s, scale_s, n_tile * BLOCK_N, BLOCK_N, cbrow, threadIdx.x - 64);
      epilogue_bar_sync();
    }
    if (warp == 2 && lane == 0) trace_ev(p, 1, tix, 45);
    const bool ok = ptx::mbar_wait(tmem_full_bar, 0, p.dbg, 3);
    ptx::tc_fence_after();
    if (warp == 2 && lane == 0) trace_ev(p, 1, tix, 46);
    // split-K staging: partial accumulators as fp32 [col][row] in this CTA's (now idle) pipeline stages
    float* stage_f = reinterpret_cast<float*>(smem);
    if (KSPLIT && krank != 0) {
      if (ok) {
#pragma unroll 1
        for (int c0 = 0; c0 < BLOCK_N; c0 += 16) {
          uint32_t rr[16];
          ptx::tc_ld_32x32b_x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, rr);
          ptx::tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; j += 4)   // [col / 4][row] float4: conflict-free 16-byte accesses on both sides
            *reinterpret_cast<float4*>(stage_f + ((c0 + j) * 128 + r * 4)) =
                make_float4(__uint_as_float(rr[j]), __uint_as_float(rr[j + 1]), __uint_as_float(rr[j + 2]), __uint_as_float(rr[j + 3]));
        }
      }
      ptx::cluster_sync_all();   // release: the leader may now read the staging through DSMEM
      mid_synced = true;
    } else {
      if (KSPLIT) { ptx::cluster_sync_all(); mid_synced = true; }   // acquire: every peer's partial tile is staged
      if (BLOCK_N == 128 && staged && p.swap_ab) {
        // ---- per-sample transposed output (V^T of the attention blocks) by operand swap: this thread's TMEM lane is
        // output channel n_tile*128 + r, the 128 columns are the tile's voxels = 256 contiguous bytes of y[n][channel][:]
        if (ok) {
          const int co = n_tile * BLOCK_N + r;
          const float bsv = (p.bias && co < p.c_out) ? __ldg(p.bias + co) : 0.f;
          const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
          const int vox0 = (d0 * p.m_h + h0) * p.m_w + w0;
#pragma unroll 1
          for (int g = 0; g < 2; ++g) {
            uint8_t* stg = smem + g * kStageBytes;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t ra[16], rb[16];
              ptx::tc_ld_32x32b_x16(trow + (uint32_t)(g * 64 + h * 32), ra);
              ptx::tc_ld_32x32b_x16(trow + (uint32_t)(g * 64 + h * 32 + 16), rb);
              ptx::tc_wait_ld();
              float v[32];
#pragma unroll
              for (int j = 0; j < 16; ++j) { v[j] = __uint_as_float(ra[j]) + bsv; v[16 + j] = __uint_as_float(rb[j]) + bsv; }
#pragma unroll
              for (int u = 0; u < 4; ++u)
                *reinterpret_cast<bf16x8*>(stg + (uint32_t)r * 128u + (uint32_t)(((h * 4 + u) ^ (r & 7)) << 4)) =
                    pack8(*reinterpret_cast<float(*)[8]>(&v[8 * u]));
            }
            ptx::fence_proxy_async();
            epilogue_bar_sync();
            if (threadIdx.x == 64) {
              ptx::tma_store_5d(&om.y[0], ptx::smem_u32(stg), vox0 + g * 64, n_tile * BLOCK_N, 0, 0, n0);
              ptx::bulk_commit_group();
            }
          }
          if (threadIdx.x == 64) ptx::bulk_wait_read_all();
        }
      } else if (BLOCK_N >= 64 && staged) {
        // ---- staged epilogue: 64-column groups -> bf16 SWIZZLE_128B tile in the (idle) pipeline stages -> one TMA store
        // per group.  Row-per-thread global stores touch 32 lines per instruction (measured ~1000 cycles per 16-column
        // chunk); the TMA store writes whole 128-byte rows and clips the ragged edges itself.
        if (ok) {
          if (staged_res) ptx::mbar_wait(res_bar, 0, p.dbg, 4);
          const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
          for (int g = 0; g < BLOCK_N / 64; ++g) {
            const int colg = n_tile * BLOCK_N + g * 64;
            if (colg >= p.c_out) break;   // CTA-uniform (c_out % 64 == 0 on this path)
            uint8_t* stg = smem + g * kStageBytes;
            const uint8_t* rs = staged_res ? res_smem + g * 16384 : nullptr;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int c0 = g * 64 + h * 32;
              uint32_t rab[2][16];
              ptx::tc_ld_32x32b_x16(trow + (uint32_t)c0, rab[0]);
              ptx::tc_ld_32x32b_x16(trow + (uint32_t)c0 + 16, rab[1]);
              ptx::tc_wait_ld();
              if (KSPLIT) add_peer_partials(rab, stage_f, c0, r, ks);
              conv_epilogue16_staged(p, rab[0], r, h * 32, n_tile * BLOCK_N + c0, has_bs ? bias_s + c0 : nullptr, cb,
                                     p.out_scale ? scale_s + c0 : nullptr, rs, stg);
              conv_epilogue16_staged(p, rab[1], r, h * 32 + 16, n_tile * BLOCK_N + c0 + 16, has_bs ? bias_s + c0 + 16 : nullptr, cb,
                                     p.out_scale ? scale_s + c0 + 16 : nullptr, rs, stg);
            }
            ptx::fence_proxy_async();
            epilogue_bar_sync();
            if (threadIdx.x == 64) {
              ptx::tma_store_5d(&om.y[parity], ptx::smem_u32(stg), colg, w0, h0, d0, n0);
              ptx::bulk_commit_group();
            }
          }
          if (threadIdx.x == 64) ptx::bulk_wait_read_all();
        }
      } else if (ok) {
#pragma unroll 1
        for (int c0 = 0; c0 < BLOCK_N; c0 += 16) {
          const int col0 = n_tile * BLOCK_N + c0;
          if (col0 >= p.c_out) break;  // warp-uniform
          uint32_t rr[1][16];
          ptx::tc_ld_32x32b_x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, rr[0]);
          ptx::tc_wait_ld();
          if (KSPLIT) add_peer_partials(rr, stage_f, c0, r, ks);
          if (!valid) continue;
          conv_epilogue16(p, rr[0], col0, n, vox, vox_per, row_off, has_bs ? bias_s + c0 : nullptr, cb,
                          p.out_scale ? scale_s + c0 : nullptr);
        }
      }
    }
  }
  if (warp == 2 && lane == 0) trace_ev(p, 1, tix, 47);
  if (KSPLIT && !mid_synced) ptx::cluster_sync_all();   // producer / MMA warps: their half of the mid-kernel barrier
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
  if (KSPLIT) ptx::cluster_sync_all();   // no CTA exits while a peer may still write / read its shared memory
  if (threadIdx.x == 0) trace_ev(p, 3, tix, 48);
}

// ------------------------------------------------------------------------------------------ host side
int pow2_ceil(int v) { int r = 1; while (r < v) r <<= 1; return r; }

struct Geometry {
  int ntaps, pad, groups, nch0, nch1, n_pad, block_n;
  int out_d, out_h, out_w, m_d, m_h, m_w;
  int box_w, box_h, box_d, box_n;
  int tiles_w, tiles_h, tiles_d, tiles_n;   // M tiles of the per-tap GEMM kernel
  long long mtiles;
  size_t ktot;
};

int compute_geometry(const b200dm_conv_desc* d, Geometry* g) {
  B2_CHECK_ARG(d, "conv: null desc");
  B2_CHECK_ARG(d->mode >= 0 && d->mode <= 2, "conv: bad mode %d", d->mode);
  B2_CHECK_ARG(d->batch > 0 && d->in_d > 0 && d->in_h > 0 && d->in_w > 0, "conv: empty input");
  B2_CHECK_ARG(d->c0 > 0 && d->c0 % 8 == 0 && d->c1 >= 0 && d->c1 % 8 == 0, "conv: C_in segments must be multiples of 8 (got %d,%d)", d->c0, d->c1);
  B2_CHECK_ARG(d->c_out > 0, "conv: c_out must be > 0");
  g->nch0 = (d->c0 + 63) / 64;
  g->nch1 = (d->c1 + 63) / 64;
  if (d->mode == B200DM_CONV_DIRECT) {
    B2_CHECK_ARG(d->ksize == 1 || d->ksize == 3 || d->ksize == 4, "conv: ksize %d unsupported", d->ksize);
    B2_CHECK_ARG(d->stride == 1 || d->stride == 2, "conv: stride %d unsupported", d->stride);
    g->ntaps = d->ksize * d->ksize * d->ksize;
    g->groups = 1;
    g->out_d = (d->in_d + d->stride - 1) / d->stride;
    g->out_h = (d->in_h + d->stride - 1) / d->stride;
    g->out_w = (d->in_w + d->stride - 1) / d->stride;
    // TF 'same': total = max((out-1)*s + k - in, 0), before = total/2.  Cubic volumes: same pad on all axes.
    B2_CHECK_ARG(d->in_d == d->in_h || d->stride == 1, "conv: strided conv needs equal D,H,W");
    int total = (g->out_w - 1) * d->stride + d->ksize - d->in_w;
    if (total < 0) total = 0;
    g->pad = total / 2;
    if (d->stride == 2) {
      int td = (g->out_d - 1) * 2 + d->ksize - d->in_d, th = (g->out_h - 1) * 2 + d->ksize - d->in_h;
      B2_CHECK_ARG((td < 0 ? 0 : td) / 2 == g->pad && (th < 0 ? 0 : th) / 2 == g->pad, "conv: strided conv needs the same 'same' padding on all axes");
    }
    g->m_d = g->out_d; g->m_h = g->out_h; g->m_w = g->out_w;
  } else if (d->mode == B200DM_CONV_PARITY) {
    B2_CHECK_ARG(d->ksize == 3 || d->ksize == 4, "conv: parity mode needs ksize 3 (upsample fold) or 4 (transposed conv)");
    g->ntaps = 8; g->groups = 8; g->pad = 0;
    g->out_d = 2 * d->in_d; g->out_h = 2 * d->in_h; g->out_w = 2 * d->in_w;
    g->m_d = d->in_d; g->m_h = d->in_h; g->m_w = d->in_w;
  } else {
    B2_CHECK_ARG(d->in_d == 1 && d->in_h == 1, "conv: batched GEMM uses in_d = in_h = 1, in_w = rows");
    B2_CHECK_ARG(d->c1 == 0, "conv: batched GEMM takes one K segment");
    g->ntaps = 1; g->groups = d->batch; g->pad = 0;
    g->out_d = 1; g->out_h = 1; g->out_w = d->in_w;
    g->m_d = 1; g->m_h = 1; g->m_w = d->in_w;
  }
  if (d->c_out <= 16) g->n_pad = 16;
  else if (d->c_out <= 32) g->n_pad = 32;
  else if (d->c_out <= 64) g->n_pad = 64;
  else g->n_pad = ((d->c_out + 127) / 128) * 128;
  g->block_n = g->n_pad < 128 ? g->n_pad : 128;
  g->ktot = (size_t)(g->nch0 + g->nch1) * g->ntaps * 64;
  // M tile box, product 128
  if (d->mode == B200DM_CONV_BATCHED_GEMM) {
    g->box_w = 128; g->box_h = 1; g->box_d = 1; g->box_n = 1;
  } else {
    int bw = pow2_ceil(g->m_w); if (bw > 8) bw = 8;
    int bh = pow2_ceil(g->m_h); if (bh > 128 / bw) bh = 128 / bw; if (bh > 16) bh = 16;
    int bd = pow2_ceil(g->m_d); if (bd > 128 / (bw * bh)) bd = 128 / (bw * bh);
    int bn = 128 / (bw * bh * bd);
    g->box_w = bw; g->box_h = bh; g->box_d = bd; g->box_n = bn;
  }
  g->tiles_w = (g->m_w + g->box_w - 1) / g->box_w; g->tiles_h = (g->m_h + g->box_h - 1) / g->box_h;
  g->tiles_d = (g->m_d + g->box_d - 1) / g->box_d; g->tiles_n = (d->batch + g->box_n - 1) / g->box_n;
  g->mtiles = (long long)g->tiles_w * g->tiles_h * g->tiles_d * g->tiles_n;
  return B200DM_OK;
}

uint16_t f32_to_bf16_rne(float f) {   // fp32 -> the library's 16-bit storage type (host side), round to nearest even
#ifdef B200DM_ACT_FP16
  const __half h = __float2half_rn(f);
  uint16_t r;
  memcpy(&r, &h, 2);
  return r;
#endif
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// ------------------------------------------------------------------------------------------ kernel selection
enum class Family { kGemm, kHalo, kHaloUp, kSweep, kStencil };   // per-tap GEMM, conv_halo.cuh, conv_halo_up.cuh, conv_sweep.cuh, conv_stencil.cuh

// Template arguments of one kernel instantiation (fields a family does not have stay 0 / false).
struct KernelKey {
  Family family;
  int block_n;                           // BLOCK_N (sweep, stencil: 0)
  int td, ns, nb, tps;                   // halo kernels: TD, slab ring depth NS, weight ring depth NB, taps per weight stage TPS
  int nstage;                            // per-tap GEMM: NSTAGE
  bool staged, pair, cg2, fuse, ksplit;  // halo kernels: STAGED, PAIR, CG2, FUSE_UPD; per-tap GEMM: KSPLIT
};
constexpr bool operator==(const KernelKey& a, const KernelKey& b) {
  return a.family == b.family && a.block_n == b.block_n && a.td == b.td && a.ns == b.ns && a.nb == b.nb && a.tps == b.tps &&
         a.nstage == b.nstage && a.staged == b.staged && a.pair == b.pair && a.cg2 == b.cg2 && a.fuse == b.fuse && a.ksplit == b.ksplit;
}

// What a plan runs: the instantiation and the runtime choices that go with it.
struct Variant {
  KernelKey key;
  bool staged_epi;   // staged epilogue: 16-bit or fp32 tile -> swizzled smem -> TMA store (halo kernels: = key.staged)
  bool swap_ab;      // per-tap GEMM: transposed store by operand swap (D^T = W X^T)
  int ksplit;        // per-tap GEMM: CTAs (one cluster) per tile, each owning a K range; 1 = off
  int dstep;         // halo kernels: output planes per tile (the pair tiles' d step is 2 with TD = 1)
  int wbox[3];       // weight-map box {channels, rows, k-blocks}; k-blocks = 0: 2-D map; channels = 0: no map
};

constexpr int kHaloNS = 6;         // slab ring depth, direct-store epilogue
constexpr int kHaloNSStaged = 5;   // staged epilogue: one slab less, the room holds the output staging tiles
// N <= 32 tiles have small weight stages and 16 KB of staging: room for the 6th slab.  With 5 (4 live per 2-plane tile) the
// issuers waited ~1000 cycles per 8000-cycle tile for the first two slabs of the next tile (tools/conv_trace.py, 128^3 32 -> 32).
constexpr int halo_ns_for(int block_n, bool staged) { return staged && block_n > 32 ? kHaloNSStaged : kHaloNS; }
constexpr int kHaloNSPair = 4;    // pair slabs are 25 KB; three per channel chunk are live
constexpr int kHaloNSWide = 4;
constexpr int kHaloNSFused = 4;   // the 16-bit staging tiles of the fused update take the room of the fifth slab

// tiles of tw x th x td voxels over the input volume, all samples
long long halo_tiles(const b200dm_conv_desc* d, int tw, int th, int td) {
  return (long long)((d->in_w + tw - 1) / tw) * ((d->in_h + th - 1) / th) * ((d->in_d + td - 1) / td) * d->batch;
}

// The kernel choice, as one ordered list of rules.  Pure: reads the descriptor, the geometry, which operands are present and
// the SM count; encodes no map and allocates nothing.
Variant select_variant(const b200dm_conv_desc* d, const Geometry& g, bool residual, bool prelu, bool chan_bias) {
  const int post_act = d->reserved[0];
  const bool transposed_store = d->reserved[1] != 0;
  const bool f32 = d->y_dtype == B200DM_F32;   // (else the 16-bit storage type)
  const bool parity = d->mode == B200DM_CONV_PARITY;
  const bool conv3 = d->mode == B200DM_CONV_DIRECT && d->ksize == 3 && d->stride == 1;
  const bool halo_ok = d->use_halo >= 0 && !transposed_store;   // use_halo = -1: per-tap GEMM kernel only
  const bool plane_8x16 = d->in_w >= 8 && d->in_h >= 16;          // planes that fill the halo kernels' 8w x 16h tile
  const bool plane_8x8 = d->in_w == 8 && d->in_h == 8;
  Variant v = {};
  KernelKey& k = v.key;
  v.ksplit = 1;
  // 1. C_out = 1, C_in = 32, 3^3 stride 1 (the vqgan_attn_cp decoder's head): HBM-bound stencil-reduce kernel instead of an
  //    N = 16 tensor-core tile (conv_stencil.cuh); bias + activation epilogue only
  if (halo_ok && conv3 && d->c_out == 1 && d->c0 == stencil::kC && d->c1 == 0 && !chan_bias && !residual && !prelu &&
      post_act == B200DM_ACT_NONE) {
    k.family = Family::kStencil;
    return v;
  }
  // 2. C_in = C_out = 32, 3^3 stride 1, 16-bit output (the decoders' 128^3 / 64^3 residual units): d-sweeping kernel with the
  //    three kd taps of an input plane as one N = 96 MMA and the weight set resident in shared memory (conv_sweep.cuh)
  if (halo_ok && conv3 && d->c_out == 32 && d->c0 == 32 && d->c1 == 0 && !f32 && !chan_bias && !prelu && plane_8x16 && d->in_d >= 2) {
    k.family = Family::kSweep;
    v.staged_epi = true;
    v.wbox[0] = 32; v.wbox[1] = 32; v.wbox[2] = 1;
    return v;
  }
  k.family = Family::kGemm;
  k.block_n = g.block_n;
  // 3. halo-reuse kernel: 3^3 stride-1 convs on volumes that fill its 8w x 16h tile
  if (halo_ok && conv3 && plane_8x16) {
    k.family = Family::kHalo;
  // 4. 8 x 8 planes (the U-Net's deepest level): pair-slab tiles, 64 output channels per CTA so that >= 128 CTAs share the
  //    weight stream; 16-bit staged output only
  } else if (halo_ok && conv3 && plane_8x8 && d->in_d >= 2 && !f32 && d->c_out % 64 == 0 && !prelu) {
    k.family = Family::kHalo;
    k.pair = true;
    k.block_n = 64;
  // 5. x2 up-convolutions (nearest-upsample + conv3, ConvT k4 s2) on low-resolution planes that fill the 8 x 16 halo tile, with an
  //    even tile count (CTA pairs).  C_out = 32 (the decoders' last ConvT, 64 -> 32 at 64^3 -> 128^3) runs N = 32 tiles with
  //    64-byte staged rows
  } else if (halo_ok && parity && plane_8x16 && d->in_d >= 2 && (d->c_out % 64 == 0 || d->c_out == 32) && !f32 && !residual &&
             !prelu && halo_tiles(d, 8, 16, 2) % 2 == 0) {
    k.family = Family::kHaloUp;
  // 6. the same on 8 x 8 low-resolution planes (8^3 -> 16^3): pair-slab tiles
  } else if (halo_ok && parity && plane_8x8 && d->in_d >= 2 && d->in_d % 2 == 0 && d->c_out % 64 == 0 && !f32 && !residual &&
             !prelu && halo_tiles(d, 8, 8, 2) % 2 == 0) {
    k.family = Family::kHaloUp;
    k.pair = true;
  }
  const bool halo = k.family != Family::kGemm;
  // 7. staged (TMA-store) epilogue: whole 64-channel groups; fp32 output (the U-Net's eps) on the halo kernels only, in 32-column
  //    groups; on the halo kernels also C_out = 32 as one 32-channel group of 64-byte rows, SWIZZLE_64B (the decoders' 128^3 convs)
  const bool n32 = halo && !k.pair && d->c_out == 32 && !f32;
  v.staged_epi = (!f32 || halo) && !transposed_store && !prelu && (d->c_out % 64 == 0 || n32) && !(parity && residual);
  // 8. per-sample transposed store by operand swap (see the kernel): tiles of whole planes inside one sample, bias only
  if (transposed_store && d->mode == B200DM_CONV_DIRECT && d->ksize == 1 && d->stride == 1 && !f32 && g.block_n == 128 &&
      g.box_n == 1 && g.box_w == g.m_w && g.box_h == g.m_h && g.m_d % g.box_d == 0 && ((long long)g.m_w * g.m_h * g.m_d) % 8 == 0 &&
      !residual && !prelu && !chan_bias && d->act == B200DM_ACT_NONE && post_act == B200DM_ACT_NONE) {
    v.swap_ab = true;
    v.staged_epi = true;
  }
  const long long sms = b2_num_sms();
  const int ntiles = g.n_pad / k.block_n;
  if (k.family == Family::kGemm) {
    const int nkb = (g.nch0 + g.nch1) * g.ntaps;
    const long long ctas = g.mtiles * (d->mode == B200DM_CONV_BATCHED_GEMM ? (d->c_out + k.block_n - 1) / k.block_n : ntiles) *
                           (parity ? 8 : 1);
    // 9. split-K: when the tile grid leaves most SMs idle and K is long, ksplit CTAs (one cluster) share a tile.  Each CTA
    //    streams its K range at the per-SM operand rate (~40 B/clk), so an under-filled grid is K-latency-bound otherwise.
    if (!transposed_store)
      while (v.ksplit < 8 && ctas * (v.ksplit * 2) <= sms && nkb / (v.ksplit * 2) >= 13) v.ksplit *= 2;   // >= 13 k-blocks per CTA: 3^3 convs only
    k.ksplit = v.ksplit > 1;
    // 10. pipeline depth 4; measured on B200: a deeper ring (6 stages at BLOCK_N=128, 8 below) does not help at BLOCK_N=128 (the
    //     operand stream is bandwidth-, not latency-bound) and hurts below 128, where 4 stages let two CTAs share an SM
    k.nstage = 4;
    // 11. short K loops (1^3 convs: 1-3 k-blocks) never fill four stages; two stages let 3-4 CTAs share an SM, which hides the
    //     per-CTA prologue / TMA latency / epilogue of these HBM-bound launches
    if (nkb <= 3 && k.block_n >= 64) k.nstage = 2;
    // 12. grids of several waves: two stages x three co-resident CTAs keep more operand bytes in flight per SM than one CTA with
    //     four stages, and hide every CTA's prologue / epilogue (measured: 16^3 128->128 parity conv 123 -> 77 us, 8^3 MLP GEMM
    //     17.5 -> 12.7 us; a single-wave split-K grid gets slower, so it keeps four stages)
    if (ctas >= 2 * sms && k.block_n >= 64 && v.ksplit <= 1) k.nstage = 2;
    // (split-K needs >= 26 k-blocks, rule 11 <= 3: no split-K plan has two stages, and no such kernel is instantiated)
    v.wbox[0] = 64; v.wbox[1] = k.block_n; v.wbox[2] = 0;
    return v;
  }
  k.staged = v.staged_epi;
  if (k.family == Family::kHaloUp) {
    // 13. up-convolutions: CTA pairs, two planes per tile, 4-tap weight stages; ring depths by BLOCK_N
    k.cg2 = true;
    v.dstep = 2;
    k.ns = k.pair ? 4 : 5;
    k.nb = k.block_n == 32 ? 4 : (k.block_n == 64 ? 3 : 2);
    k.tps = 4;
  } else {
    // 14. planes per tile: 2 (weight stage shared by two planes, two MMA issuer warps) unless that costs a wave
    const long long cost2 = (halo_tiles(d, 8, 16, 2) * ntiles + sms - 1) / sms * 2, cost1 = (halo_tiles(d, 8, 16, 1) * ntiles + sms - 1) / sms;
    const int td = d->in_d >= 2 && cost2 <= cost1 ? 2 : 1;
    v.dstep = k.pair ? 2 : td;   // (pair tiles: d step 2, one accumulator)
    k.td = k.pair ? 1 : td;
    // 15. weight-ring depth / taps per stage by BLOCK_N (smem: 6 slabs x 23 KB + NB x TPS x BLOCK_N x 128 B <= 227 KB)
    k.nb = k.block_n == 64 ? 3 : 4;
    k.tps = k.block_n >= 128 ? 1 : 3;
    k.ns = k.pair ? kHaloNSPair : halo_ns_for(k.block_n, k.staged);
    // 16. BLOCK_N = 128 with the staged epilogue: one-tap weight stages hold only 8 MMAs (4 per issuer warp) and the per-stage
    //     barrier round trip (~200 cycles) made those convs issue-bound (45 % of the MMA floor); 3-tap stages x 2 fit once the
    //     slab ring is the 4 slabs a channel chunk needs (the next chunk's slab i reloads as soon as slab i is released).
    if (!k.pair && k.block_n == 128 && k.staged) { k.nb = 2; k.tps = 3; k.ns = kHaloNSWide; }
    // 17. CTA pairs (cta_group::2) for every staged halo configuration with 64- or 128-channel tiles, and for N = 32 convs with at
    //     least two channel chunks (the U-Net's input conv, 256 -> 32, direct stores): needs an even tile count per n-tile so that
    //     the two CTAs of a pair always work on the same n-tile and run the same number of tiles.  Short-K N = 32 convs (one
    //     channel chunk) stay single-CTA: with direct stores pairing couples two epilogues (measured 4.18 -> 4.79 ms), staged it
    //     gained 3.79 -> 3.74 ms only.
    const bool cg2_n32 = k.block_n == 32 && !k.pair && td == 2 && g.nch0 + g.nch1 >= 2;
    const bool cg2_wide = (k.block_n == 64 || k.block_n == 128) && k.staged && (k.pair || td == 2 || k.block_n == 128);
    if ((cg2_wide || cg2_n32) && halo_tiles(d, 8, k.pair ? 8 : 16, v.dstep) % 2 == 0) {
      k.cg2 = true;
      k.nb = cg2_n32 ? 4 : 3;
      k.tps = 3;
      k.ns = k.pair ? kHaloNSPair : halo_ns_for(k.block_n, k.staged);
    }
  }
  // packed weights viewed as {64, rows, k-blocks}: one box = TPS consecutive taps of this CTA's rows (a CTA pair: half each)
  v.wbox[0] = 64; v.wbox[1] = k.cg2 ? k.block_n / 2 : k.block_n; v.wbox[2] = k.tps;
  return v;
}

// NDHWC tensor of c channels and extent (w, h, d, n) as a 5-D TMA map.  step: voxels per map coordinate along W, H, D (2: one
// output parity of a x2 up-convolution, the map spans half the extent); estride: TMA element stride (a stride-2 conv's
// input); dh_order: dims listed (C, W, D, H, N), so that a box lands as rows [h][d][w] (pair slabs).
int encode_act(EncodeTiledFn enc, CUtensorMap* m, const char* what, const void* base, CUtensorMapDataType dt, int c, int w, int h,
               int d, int n, const cuuint32_t (&box)[5], CUtensorMapSwizzle swz, int step = 1, cuuint32_t estride = 1,
               bool dh_order = false) {
  const cuuint64_t sw = (cuuint64_t)c * (dt == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? 4 : 2), sh = sw * w, sd = sh * h, sn = sd * d;
  cuuint64_t dims[5] = {(cuuint64_t)c, (cuuint64_t)(w / step), (cuuint64_t)(h / step), (cuuint64_t)(d / step), (cuuint64_t)n};
  cuuint64_t strides[4] = {sw * step, sh * step, sd * step, sn};
  if (dh_order) { std::swap(dims[2], dims[3]); std::swap(strides[1], strides[2]); }
  const cuuint32_t es[5] = {1, estride, estride, estride, 1};
  const CUresult r = enc(m, dt, 5, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    b200dm_set_error("cuTensorMapEncodeTiled(%s) failed: %d (C=%d dims %d,%d,%d,%d box %u,%u,%u,%u)", what, (int)r, c, w, h, d, n,
                     box[1], box[2], box[3], box[4]);
    return B200DM_ERR_CUDA;
  }
  return B200DM_OK;
}

// packed weights [groups * n_pad rows][ktot / 64 k-blocks][64] as the 3-D view {64, rows, k-blocks}; a box row of 64 (32)
// channels is one 128-byte (64-byte) swizzle span.  ktot: the row length (g.ktot, or longer with a folded shortcut's k-blocks)
int encode_weights3(EncodeTiledFn enc, CUtensorMap* m, const void* w, const Geometry& g, const int (&box)[3], size_t ktot) {
  const cuuint64_t dims[3] = {64, (cuuint64_t)g.groups * g.n_pad, (cuuint64_t)(ktot / 64)};
  const cuuint64_t strides[2] = {(cuuint64_t)ktot * 2, 128};
  const cuuint32_t b[3] = {(cuuint32_t)box[0], (cuuint32_t)box[1], (cuuint32_t)box[2]}, es[3] = {1, 1, 1};
  const CUresult r = enc(m, kTmapAct16, 3, const_cast<void*>(w), dims, strides, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         box[0] == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { b200dm_set_error("cuTensorMapEncodeTiled(B) failed: %d (box %d,%d,%d)", (int)r, box[0], box[1], box[2]); return B200DM_ERR_CUDA; }
  return B200DM_OK;
}

struct Instance;

}  // namespace

struct b200dm_conv_plan {
  b200dm_conv_desc desc;
  Geometry g;
  Variant v;
  const Instance* inst;   // the instantiation v.key names
  ConvParams p;
  CUtensorMap mapA0, mapA1, mapB;
  ConvOutMaps om;
  CUtensorMap mapS;       // stencil / sweep kernels: the input (mapB = the sweep kernel's weights, om.y[0] its output)
  CUtensorMap mapSc0, mapSc1;   // halo kernel: the two input segments of a folded 1^3 shortcut (b200dm_conv_plan_set_shortcut)
  stencil::Params sp;
  sweep::Params wp;
  dim3 grid;
  size_t smem;
  double flops;
};

static int* g_dbg_flag = nullptr;
static int ensure_dbg_flag() {
  if (!g_dbg_flag) {
    B2_CHECK_CUDA(cudaMalloc(&g_dbg_flag, sizeof(int)));
    B2_CHECK_CUDA(cudaMemset(g_dbg_flag, 0, sizeof(int)));
  }
  return B200DM_OK;
}

int* b200dm_dbg_flag_ptr() { return ensure_dbg_flag() == B200DM_OK ? g_dbg_flag : nullptr; }

extern "C" int b200dm_debug_flag_read_reset(int32_t* flag_out) {
  B2_CHECK_ARG(flag_out, "debug_flag: null");
  *flag_out = 0;
  if (!g_dbg_flag) return B200DM_OK;
  B2_CHECK_CUDA(cudaMemcpy(flag_out, g_dbg_flag, sizeof(int), cudaMemcpyDeviceToHost));
  B2_CHECK_CUDA(cudaMemset(g_dbg_flag, 0, sizeof(int)));
  return B200DM_OK;
}

extern "C" size_t b200dm_conv_packed_weight_bytes(const b200dm_conv_desc* d) {
  Geometry g;
  if (compute_geometry(d, &g) != B200DM_OK) return 0;
  if (d->mode == B200DM_CONV_BATCHED_GEMM) return 0;
  return (size_t)g.groups * g.n_pad * g.ktot * 2;
}

extern "C" int b200dm_conv_pack_weights(const b200dm_conv_desc* d, const float* w, int32_t transposed, void* packed) {
  Geometry g;
  int rc = compute_geometry(d, &g);
  if (rc) return rc;
  B2_CHECK_ARG(w && packed, "conv_pack_weights: null pointer");
  B2_CHECK_ARG(d->mode != B200DM_CONV_BATCHED_GEMM, "conv_pack_weights: batched GEMM has no packed weights");
  const int k = d->ksize, cin = d->c0 + d->c1, cout = d->c_out;
  uint16_t* out = reinterpret_cast<uint16_t*>(packed);
  memset(out, 0, (size_t)g.groups * g.n_pad * g.ktot * 2);
  // Keras kernel index: ((kd*k + kh)*k + kw) * cin*cout + (transposed ? co*cin + ci : ci*cout + co)
  auto W = [&](int kd, int kh, int kw, int ci, int co) -> float {
    const size_t base = ((size_t)(kd * k + kh) * k + kw) * (size_t)cin * cout;
    return transposed ? w[base + (size_t)co * cin + ci] : w[base + (size_t)ci * cout + co];
  };
  const int nch = g.nch0 + g.nch1;
  for (int grp = 0; grp < g.groups; ++grp) {
    const int pw = grp & 1, ph = (grp >> 1) & 1, pd = (grp >> 2) & 1;
    for (int co = 0; co < cout; ++co) {
      uint16_t* row = out + ((size_t)grp * g.n_pad + co) * g.ktot;
      for (int ch = 0; ch < nch; ++ch) {
        for (int tap = 0; tap < g.ntaps; ++tap) {
          for (int c = 0; c < 64; ++c) {
            int ci;
            if (ch < g.nch0) { ci = ch * 64 + c; if (ci >= d->c0) continue; }
            else { ci = (ch - g.nch0) * 64 + c; if (ci >= d->c1) continue; ci += d->c0; }
            float v = 0.f;
            if (d->mode == B200DM_CONV_DIRECT) {
              v = W(tap / (k * k), (tap / k) % k, tap % k, ci, co);
            } else {
              const int tw = tap & 1, th = (tap >> 1) & 1, tdp = (tap >> 2) & 1;
              if (k == 3) {
                // nearest-upsample fold: parity 0: slot0 (offset -1) <- {k0}, slot1 (offset 0) <- {k1,k2};
                //                        parity 1: slot0 (offset 0) <- {k0,k1}, slot1 (offset +1) <- {k2}
                auto lo = [](int par, int slot) { return par == 0 ? (slot == 0 ? 0 : 1) : (slot == 0 ? 0 : 2); };
                auto hi = [](int par, int slot) { return par == 0 ? (slot == 0 ? 0 : 2) : (slot == 0 ? 1 : 2); };
                double acc = 0.0;
                for (int kd = lo(pd, tdp); kd <= hi(pd, tdp); ++kd)
                  for (int kh = lo(ph, th); kh <= hi(ph, th); ++kh)
                    for (int kw = lo(pw, tw); kw <= hi(pw, tw); ++kw) acc += (double)W(kd, kh, kw, ci, co);
                v = (float)acc;
              } else {
                // transposed conv k4 s2 'same': out[2m+p] = sum_off in[m+off] * w[p + 1 - 2*off], off = slot - 1 + p
                auto kk = [](int par, int slot) { return par + 1 - 2 * (slot - 1 + par); };
                v = W(kk(pd, tdp), kk(ph, th), kk(pw, tw), ci, co);
              }
            }
            row[((size_t)ch * g.ntaps + tap) * 64 + c] = f32_to_bf16_rne(v);
          }
        }
      }
    }
  }
  return B200DM_OK;
}

namespace {

// ------------------------------------------------------------------------------------------ kernel instantiations
// Kernel arguments, by kernel signature.
template <typename... KArgs, typename... Args>
cudaError_t launch_plan(void (*k)(KArgs...), const b200dm_conv_plan* pl, unsigned threads, cudaStream_t s, Args... args) {
  const unsigned cluster = pl->v.key.cg2 ? 2u : (unsigned)pl->v.ksplit;
  return b2_launch_cluster(k, pl->grid, dim3(threads), cluster, pl->smem, s, args...);
}
// per-tap GEMM, halo up-convolution
cudaError_t launch_args(void (*k)(CUtensorMap, CUtensorMap, CUtensorMap, ConvOutMaps, ConvParams), const b200dm_conv_plan* pl,
                        unsigned threads, cudaStream_t s) {
  return launch_plan(k, pl, threads, s, pl->mapA0, pl->mapA1, pl->mapB, pl->om, pl->p);
}
// halo kernel: output map (the fused update: x_{t-1}) and its 16-bit copy, shortcut input segments
cudaError_t launch_args(void (*k)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, ConvParams),
                        const b200dm_conv_plan* pl, unsigned threads, cudaStream_t s) {
  return launch_plan(k, pl, threads, s, pl->mapA0, pl->mapA1, pl->mapB, pl->om.y[0], pl->om.y[1], pl->mapSc0, pl->mapSc1, pl->p);
}
// sweep kernel: input, weights, output, residual (a valid map either way: unused without a residual)
cudaError_t launch_args(void (*k)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, ConvParams, sweep::Params),
                        const b200dm_conv_plan* pl, unsigned threads, cudaStream_t s) {
  return launch_plan(k, pl, threads, s, pl->mapS, pl->mapB, pl->om.y[0], pl->p.residual ? pl->om.r : pl->om.y[0], pl->p, pl->wp);
}
cudaError_t launch_args(void (*k)(CUtensorMap, stencil::Params), const b200dm_conv_plan* pl, unsigned threads, cudaStream_t s) {
  return launch_plan(k, pl, threads, s, pl->mapS, pl->sp);
}

struct Instance {
  KernelKey key;
  unsigned threads;
  size_t smem, smem_res;   // dynamic shared memory; smem_res: with the per-tap GEMM kernel's staged residual tile
  int (*launch)(const b200dm_conv_plan*, cudaStream_t);
  cudaError_t (*set_max_smem)(int bytes);
};

template <auto K>
int launch(const b200dm_conv_plan* pl, cudaStream_t s) {
  B2_CHECK_CUDA(launch_args(K, pl, pl->inst->threads, s));
  return B200DM_OK;
}
template <auto K>
cudaError_t set_max_smem(int bytes) { return cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); }

template <auto K>
constexpr Instance instance(KernelKey key, unsigned threads, size_t smem, size_t smem_res) {
  return {key, threads, smem, smem_res, &launch<K>, &set_max_smem<K>};
}
template <int BLOCK_N, int NSTAGE, bool KSPLIT>
constexpr Instance gemm() {
  using L = GemmSmem<BLOCK_N, NSTAGE>;
  return instance<conv_igemm_kernel<BLOCK_N, NSTAGE, KSPLIT>>(
      {Family::kGemm, BLOCK_N, 0, 0, 0, 0, NSTAGE, false, false, false, false, KSPLIT}, kThreads, L::bytes(false), L::bytes(true));
}
template <int BLOCK_N, int TD, int NS, int NB, int TPS, bool STAGED, bool PAIR = false, bool CG2 = false, bool FUSE_UPD = false>
constexpr Instance halo_conv() {
  constexpr size_t kBytes = halo::Smem<BLOCK_N, NS, NB, TPS, STAGED, PAIR, CG2, FUSE_UPD>::kBytes;
  return instance<halo::conv_halo_kernel<BLOCK_N, TD, NS, NB, TPS, STAGED, PAIR, CG2, FUSE_UPD>>(
      {Family::kHalo, BLOCK_N, TD, NS, NB, TPS, 0, STAGED, PAIR, CG2, FUSE_UPD, false}, FUSE_UPD ? halo::kThreadsFused : halo::kThreads,
      kBytes, kBytes);
}
template <int BLOCK_N, int NS, int NB, bool PAIR = false>
constexpr Instance halo_up() {
  constexpr size_t kBytes = halo::UpSmem<BLOCK_N, NS, NB, PAIR>::kBytes;
  return instance<halo::conv_halo_up_kernel<BLOCK_N, NS, NB, PAIR>>(
      {Family::kHaloUp, BLOCK_N, 0, NS, NB, 4, 0, true, PAIR, true, false, false}, halo::kThreads, kBytes, kBytes);
}

// Every conv kernel instantiation, each a configuration select_variant can return.  A key without an entry is an error.
constexpr Instance kInstances[] = {
    instance<stencil::conv_stencil_c1_kernel>({Family::kStencil}, stencil::kThreads, stencil::kSmem, stencil::kSmem),
    instance<sweep::conv_sweep32_kernel>({Family::kSweep}, sweep::kThreads, sweep::kSmem, sweep::kSmem),
    gemm<16, 4, false>(), gemm<32, 4, false>(), gemm<64, 4, false>(), gemm<128, 4, false>(),
    gemm<64, 2, false>(), gemm<128, 2, false>(),
    gemm<16, 4, true>(), gemm<32, 4, true>(), gemm<64, 4, true>(), gemm<128, 4, true>(),
    // one CTA per tile
    halo_conv<16, 1, kHaloNS, 4, 3, false>(), halo_conv<16, 2, kHaloNS, 4, 3, false>(),
    halo_conv<32, 1, kHaloNS, 4, 3, false>(), halo_conv<32, 2, kHaloNS, 4, 3, false>(),
    halo_conv<32, 1, kHaloNS, 4, 3, true>(), halo_conv<32, 2, kHaloNS, 4, 3, true>(),
    halo_conv<64, 1, kHaloNS, 3, 3, false>(), halo_conv<64, 2, kHaloNS, 3, 3, false>(),
    halo_conv<64, 1, kHaloNSStaged, 3, 3, true>(), halo_conv<64, 2, kHaloNSStaged, 3, 3, true>(),
    halo_conv<128, 1, kHaloNS, 4, 1, false>(), halo_conv<128, 2, kHaloNS, 4, 1, false>(),
    halo_conv<128, 1, kHaloNSWide, 2, 3, true>(), halo_conv<128, 2, kHaloNSWide, 2, 3, true>(),
    halo_conv<64, 1, kHaloNSPair, 3, 3, true, true>(),
    // CTA pairs
    halo_conv<32, 2, kHaloNS, 4, 3, false, false, true>(), halo_conv<32, 2, kHaloNS, 4, 3, true, false, true>(),
    halo_conv<64, 2, kHaloNSStaged, 3, 3, true, false, true>(),
    halo_conv<128, 1, kHaloNSStaged, 3, 3, true, false, true>(), halo_conv<128, 2, kHaloNSStaged, 3, 3, true, false, true>(),
    halo_conv<64, 1, kHaloNSPair, 3, 3, true, true, true>(),
    halo_conv<128, 1, kHaloNSFused, 3, 3, true, false, true, true>(), halo_conv<128, 2, kHaloNSFused, 3, 3, true, false, true, true>(),
    halo_up<32, 5, 4>(), halo_up<64, 5, 3>(), halo_up<128, 5, 2>(), halo_up<64, 4, 3, true>(), halo_up<128, 4, 2, true>(),
};

// Binds the instantiation of `v` to the plan: its launcher and shared-memory size, and the kernel's opt-in shared-memory limit.
// The plan is left unchanged on failure.
int bind_kernel(b200dm_conv_plan* pl, const Variant& v) {
  const Instance* inst = nullptr;
  for (const Instance& i : kInstances)
    if (i.key == v.key) { inst = &i; break; }
  if (!inst) {
    b200dm_set_error("conv_plan: no kernel instantiation for family %d, BLOCK_N %d", (int)v.key.family, v.key.block_n);
    return B200DM_ERR_UNSUPPORTED;
  }
  if (inst->smem_res > kMaxDynamicSmem) { b200dm_set_error("conv_plan: %zu bytes of shared memory", inst->smem_res); return B200DM_ERR_UNSUPPORTED; }
  B2_CHECK_CUDA(inst->set_max_smem((int)inst->smem_res));
  pl->v = v;
  pl->inst = inst;
  pl->smem = v.staged_epi && pl->p.residual ? inst->smem_res : inst->smem;
  return B200DM_OK;
}

// Tensor maps and launch parameters of a plan whose pl->v is selected.
int setup_plan(b200dm_conv_plan* pl, EncodeTiledFn enc, const void* x0, const void* x1, const void* w_packed, const float* bias,
               const float* chan_bias, const int32_t* t_dev, const void* residual, const void* prelu_alpha, void* y) {
  const b200dm_conv_desc* d = &pl->desc;
  const Geometry& g = pl->g;
  Variant& v = pl->v;
  const KernelKey& k = v.key;
  ConvParams& p = pl->p;
  const long long sms = b2_num_sms();
  int rc;
  if (k.family == Family::kStencil) {
    rc = encode_act(enc, &pl->mapS, "stencil X", x0, kTmapAct16, d->c0, d->in_w, d->in_h, d->in_d, d->batch,
                    {(cuuint32_t)stencil::kC, (cuuint32_t)stencil::kHW, (cuuint32_t)stencil::kHH, 1, 1}, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    stencil::Params& sp = pl->sp;
    sp.batch = d->batch; sp.D = d->in_d; sp.H = d->in_h; sp.W = d->in_w;
    sp.tiles_h = (d->in_h + stencil::kTH - 1) / stencil::kTH; sp.tiles_w = (d->in_w + stencil::kTW - 1) / stencil::kTW;
    // d ranges: enough work items for ~6 per resident CTA (two CTAs per SM), each range >= 8 planes (2 halo planes per range)
    const long long cols = (long long)d->batch * sp.tiles_h * sp.tiles_w, ctas = 2 * sms;
    int dsplit = 1;
    while (cols * dsplit < 6 * ctas && d->in_d / (dsplit * 2) >= 8) dsplit *= 2;
    sp.dlen = (d->in_d + dsplit - 1) / dsplit; sp.dsplit = (d->in_d + sp.dlen - 1) / sp.dlen;
    sp.items = (int)(cols * sp.dsplit);
    sp.w = (const act_t*)w_packed; sp.bias = bias; sp.act = d->act; sp.y_f32 = d->y_dtype == B200DM_F32; sp.y = y; sp.dbg = g_dbg_flag;
    pl->grid = dim3((unsigned)(sp.items < ctas ? sp.items : ctas), 1, 1);
    return B200DM_OK;
  }
  if (k.family == Family::kSweep) {
    const cuuint32_t boxy[5] = {32, 8, 16, 1, 1};
    rc = encode_act(enc, &pl->mapS, "sweep X", x0, kTmapAct16, 32, d->in_w, d->in_h, d->in_d, d->batch, {32, 10, 18, 2, 1},
                    CU_TENSOR_MAP_SWIZZLE_64B);
    if (!rc) rc = encode_act(enc, &pl->om.y[0], "sweep Y", y, kTmapAct16, 32, d->in_w, d->in_h, d->in_d, d->batch, boxy, CU_TENSOR_MAP_SWIZZLE_64B);
    if (!rc) rc = encode_weights3(enc, &pl->mapB, w_packed, g, v.wbox, g.ktot);
    if (!rc && residual)
      rc = encode_act(enc, &pl->om.r, "sweep residual", residual, kTmapAct16, 32, d->in_w, d->in_h, d->in_d, d->batch, boxy, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    sweep::Params& wp = pl->wp;
    wp.D = d->in_d; wp.H = d->in_h; wp.W = d->in_w; wp.batch = d->batch;
    wp.tiles_w = (d->in_w + 7) / 8; wp.tiles_h = (d->in_h + 15) / 16;
    const long long cols = (long long)d->batch * wp.tiles_w * wp.tiles_h, ctas = sms;
    int dsplit = 1;
    while (cols * dsplit < 6 * ctas && d->in_d / (dsplit * 2) >= 8) dsplit *= 2;   // >= ~6 items per CTA, d ranges of >= 8 planes
    wp.dlen = (d->in_d + dsplit - 1) / dsplit; wp.dsplit = (d->in_d + wp.dlen - 1) / wp.dlen;
    wp.items = (int)(cols * wp.dsplit);
    p.batch = d->batch; p.in_d = p.out_d = d->in_d; p.in_h = p.out_h = d->in_h; p.in_w = p.out_w = d->in_w;
    p.c_out = 32; p.n_pad = 32; p.act = d->act; p.post_act = d->reserved[0];
    p.bias = bias; p.residual = (const act_t*)residual; p.y = y; p.dbg = g_dbg_flag; p.tma_epi = 1;
    pl->grid = dim3((unsigned)(wp.items < ctas ? wp.items : ctas), 1, 1);
    return B200DM_OK;
  }
  // per-tap GEMM and halo kernels
  if (g.mtiles > 0x7fffffffLL) { b200dm_set_error("conv_plan_create: too many tiles"); return B200DM_ERR_INVALID; }
  const bool halo = k.family != Family::kGemm, up = k.family == Family::kHaloUp, f32 = d->y_dtype == B200DM_F32;
  const bool parity = d->mode == B200DM_CONV_PARITY;
  const int st = d->mode == B200DM_CONV_DIRECT ? d->stride : 1;
  {  // activations: the GEMM tile's box shifted per tap, or one halo d-plane slab (pair slab: {64, 10, 2, 10, 1} as rows [h][d][w])
    const cuuint32_t box[5] = {64, (cuuint32_t)(k.pair ? 10 : halo ? 10 : g.box_w * st), (cuuint32_t)(k.pair ? 2 : halo ? 18 : g.box_h * st),
                               (cuuint32_t)(k.pair ? 10 : halo ? 1 : g.box_d * st), (cuuint32_t)(halo ? 1 : g.box_n)};
    rc = encode_act(enc, &pl->mapA0, "A", x0, kTmapAct16, d->c0, d->in_w, d->in_h, d->in_d, d->batch, box, CU_TENSOR_MAP_SWIZZLE_128B, 1,
                    (cuuint32_t)st, k.pair);
    if (!rc) rc = encode_act(enc, &pl->mapA1, "A", d->c1 > 0 ? x1 : x0, kTmapAct16, d->c1 > 0 ? d->c1 : d->c0, d->in_w, d->in_h, d->in_d,
                             d->batch, box, CU_TENSOR_MAP_SWIZZLE_128B, 1, (cuuint32_t)st, k.pair);
    if (rc) return rc;
  }
  if (halo) {
    rc = encode_weights3(enc, &pl->mapB, w_packed, g, v.wbox, g.ktot);
    if (rc) return rc;
  } else {
    // packed [group][n_pad rows][K]; batched GEMM: B is a raw activation tensor [batch][c_out rows][K = c0] whose rows beyond c_out
    // of a sample alias the next sample (masked by the epilogue's col < c_out), K beyond c0 is zero-filled by TMA
    const bool bg = d->mode == B200DM_CONV_BATCHED_GEMM;
    const cuuint64_t dims[2] = {bg ? (cuuint64_t)d->c0 : (cuuint64_t)g.ktot, bg ? (cuuint64_t)d->batch * d->c_out : (cuuint64_t)g.groups * g.n_pad};
    const cuuint64_t strides[1] = {dims[0] * 2};
    const cuuint32_t box[2] = {(cuuint32_t)v.wbox[0], (cuuint32_t)v.wbox[1]}, es[2] = {1, 1};
    const CUresult r = enc(&pl->mapB, kTmapAct16, 2, const_cast<void*>(w_packed), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { b200dm_set_error("cuTensorMapEncodeTiled(B) failed: %d", (int)r); return B200DM_ERR_CUDA; }
  }
  if (v.swap_ab) {
    // per-sample transposed output [n][channel][voxel]: one box = 64 voxels x 128 channels.  Should the encode fail, the plan
    // keeps the scalar transposed store.
    const cuuint64_t Lv = (cuuint64_t)g.m_w * g.m_h * g.m_d;
    const cuuint64_t dims[5] = {Lv, (cuuint64_t)d->c_out, 1, 1, (cuuint64_t)d->batch};
    const cuuint64_t strides[4] = {Lv * 2, Lv * d->c_out * 2, Lv * d->c_out * 2, Lv * d->c_out * 2};
    const cuuint32_t box[5] = {64, 128, 1, 1, 1}, es[5] = {1, 1, 1, 1, 1};
    if (enc(&pl->om.y[0], kTmapAct16, 5, y, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      v.swap_ab = v.staged_epi = false;
  } else if (v.staged_epi) {
    // output tile of the GEMM kernel, one output plane of the halo kernels (pair: 8w x 2d x 8h); 64-channel groups of 128-byte
    // rows, fp32: 32-channel groups; C_out = 32 on the halo kernels: one group of 64-byte rows
    const bool group32 = k.block_n == 32;
    const CUtensorMapDataType dt = f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : kTmapAct16;
    const CUtensorMapSwizzle swz = group32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
    const cuuint32_t box[5] = {f32 || group32 ? 32u : 64u, (cuuint32_t)(halo ? 8 : g.box_w), (cuuint32_t)(k.pair ? 2 : halo ? 16 : g.box_h),
                               (cuuint32_t)(k.pair ? 8 : halo ? 1 : g.box_d), (cuuint32_t)(halo ? 1 : g.box_n)};
    const int ps = parity ? 2 : 1;   // output voxel stride of one M-space step; one map per output parity
    for (int q = 0; q < (parity ? 8 : 1) && !rc; ++q) {
      const size_t off = ((size_t)((q >> 2) & 1) * g.out_h * g.out_w + (size_t)((q >> 1) & 1) * g.out_w + (size_t)(q & 1)) * d->c_out * (f32 ? 4 : 2);
      rc = encode_act(enc, &pl->om.y[q], "Y", (const char*)y + (parity ? off : 0), dt, d->c_out, g.out_w, g.out_h, g.out_d, d->batch, box,
                      swz, ps, 1, k.pair);
    }
    if (!rc && residual && !halo)   // (the halo kernels read the residual into registers)
      rc = encode_act(enc, &pl->om.r, "residual", residual, dt, d->c_out, g.out_w, g.out_h, g.out_d, d->batch, box, swz);
    if (rc) return rc;
  }
  p.mode = d->mode; p.batch = d->batch;
  p.in_d = d->in_d; p.in_h = d->in_h; p.in_w = d->in_w;
  p.out_d = g.out_d; p.out_h = g.out_h; p.out_w = g.out_w;
  p.m_d = g.m_d; p.m_h = g.m_h; p.m_w = g.m_w;
  p.box_w = g.box_w; p.box_h = g.box_h; p.box_d = g.box_d; p.box_n = g.box_n;
  p.tiles_w = g.tiles_w; p.tiles_h = g.tiles_h; p.tiles_d = g.tiles_d; p.tiles_n = g.tiles_n;
  p.nch0 = g.nch0; p.nch1 = g.nch1; p.ntaps = g.ntaps; p.ksize = d->ksize; p.stride = st; p.pad = g.pad;
  p.ksteps0_last = ((d->c0 - (g.nch0 - 1) * 64) + 15) / 16;
  p.ksteps1_last = d->c1 > 0 ? ((d->c1 - (g.nch1 - 1) * 64) + 15) / 16 : 4;
  p.c_out = d->c_out; p.n_pad = d->mode == B200DM_CONV_BATCHED_GEMM ? d->c_out : g.n_pad;
  p.act = d->act; p.post_act = d->reserved[0]; p.y_f32 = f32; p.transposed_store = d->reserved[1];
  p.chan_bias_rows = d->chan_bias_rows;
  p.bias = bias; p.chan_bias = chan_bias; p.t_dev = t_dev;
  p.residual = (const act_t*)residual; p.prelu_alpha = (const act_t*)prelu_alpha;
  p.y = y; p.dbg = g_dbg_flag;
  p.tma_epi = v.staged_epi; p.swap_ab = v.swap_ab; p.ksplit = v.ksplit;
  const int ntiles = d->mode == B200DM_CONV_BATCHED_GEMM ? (d->c_out + k.block_n - 1) / k.block_n : g.n_pad / k.block_n;
  if (!halo) {
    pl->grid = dim3((unsigned)(g.mtiles * v.ksplit), (unsigned)ntiles, parity ? 8 : 1);
    return B200DM_OK;
  }
  // persistent halo kernels: at most one CTA per SM (whole pairs) walks the tile list
  p.tiles_w = (d->in_w + 7) / 8; p.tiles_h = k.pair ? (d->in_h + 7) / 8 : (d->in_h + 15) / 16; p.tiles_d = (d->in_d + v.dstep - 1) / v.dstep;
  p.tiles_n = d->batch;
  const long long per = (long long)p.tiles_w * p.tiles_h * p.tiles_d * p.tiles_n;
  p.halo_td = v.dstep; p.halo_tiles_per_ntile = (int)per; p.halo_ntn = ntiles; p.halo_total_tiles = (int)(per * ntiles * (up ? 8 : 1));
  int ctas = (int)sms;
  if (ctas > p.halo_total_tiles) ctas = p.halo_total_tiles;
  if (k.cg2) ctas &= ~1;
  pl->grid = dim3((unsigned)ctas, 1, 1);
  return B200DM_OK;
}

}  // namespace

extern "C" int b200dm_conv_plan_create(const b200dm_conv_desc* d, const void* x0, const void* x1, const void* w_packed,
                                       const float* bias, const float* chan_bias, const int32_t* t_dev,
                                       const void* residual, const void* prelu_alpha, void* y,
                                       b200dm_conv_plan** out) {
  B2_CHECK_ARG(out, "conv_plan_create: null out");
  *out = nullptr;
  Geometry g;
  int rc = compute_geometry(d, &g);
  if (rc) return rc;
  B2_CHECK_ARG(x0 && w_packed && y, "conv_plan_create: null tensor pointer");
  B2_CHECK_ARG((d->c1 > 0) == (x1 != nullptr), "conv_plan_create: x1 must be given iff c1 > 0");
  B2_CHECK_ARG(d->y_dtype == B200DM_BF16 || d->y_dtype == B200DM_F32, "conv_plan_create: bad y dtype");
  B2_CHECK_ARG(((uintptr_t)x0 & 15) == 0 && ((uintptr_t)w_packed & 15) == 0 && ((uintptr_t)y & 15) == 0, "conv_plan_create: pointers must be 16-byte aligned");
  EncodeTiledFn enc = b2_encode_tiled_fn();
  if (!enc) { b200dm_set_error("conv_plan_create: cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return B200DM_ERR_CUDA; }
  rc = ensure_dbg_flag();
  if (rc) return rc;

  std::unique_ptr<b200dm_conv_plan> pl(new (std::nothrow) b200dm_conv_plan());
  B2_CHECK_ARG(pl, "conv_plan_create: out of memory");
  pl->desc = *d;
  pl->g = g;
  pl->v = select_variant(d, g, residual != nullptr, prelu_alpha != nullptr, chan_bias != nullptr);
  rc = setup_plan(pl.get(), enc, x0, x1, w_packed, bias, chan_bias, t_dev, residual, prelu_alpha, y);
  if (!rc) rc = bind_kernel(pl.get(), pl->v);
  if (rc) return rc;
  // algorithmic FLOPs (SURVEY 8d): 2*k^3*Cin*Cout*B*out_voxels; convT: 2*64*Cin*Cout*B*in_voxels; GEMM: 2*M*N*K
  if (d->mode == B200DM_CONV_PARITY)
    pl->flops = d->ksize == 3 ? 2.0 * 27 * (d->c0 + d->c1) * d->c_out * (double)d->batch * g.out_d * g.out_h * g.out_w
                              : 2.0 * 64 * (d->c0 + d->c1) * d->c_out * (double)d->batch * d->in_d * d->in_h * d->in_w;
  else
    pl->flops = 2.0 * g.ntaps * (d->c0 + d->c1) * d->c_out * (double)d->batch * g.out_d * g.out_h * g.out_w;
  *out = pl.release();
  return B200DM_OK;
}

extern "C" int b200dm_conv_plan_run(b200dm_conv_plan* pl, void* stream) {
  B2_CHECK_ARG(pl, "conv_plan_run: null plan");
  return pl->inst->launch(pl, (cudaStream_t)stream);
}

extern "C" void b200dm_conv_plan_destroy(b200dm_conv_plan* p) { delete p; }

// tuning aid: device buffer of 4 * 2048 int64 receiving CTA 0's per-role timeline ((clock64 << 8) | tag); nullptr = off
extern "C" int b200dm_conv_plan_set_trace(b200dm_conv_plan* p, void* trace) {
  B2_CHECK_ARG(p, "conv_plan_set_trace: null plan");
  p->p.trace = (long long*)trace;
  return B200DM_OK;
}

extern "C" double b200dm_conv_plan_flops(const b200dm_conv_plan* p) { return p ? p->flops : 0.0; }

extern "C" int b200dm_conv_plan_set_fused_update(b200dm_conv_plan* pl, const b200dm_update_desc* u, const float* x_t, float* x_prev,
                                                 void* x_prev_16) {
  B2_CHECK_ARG(pl && u && x_t && x_prev && x_prev_16, "conv_plan_set_fused_update: null argument");
  const b200dm_conv_desc* d = &pl->desc;
  const ConvParams& p = pl->p;
  const KernelKey& k = pl->v.key;
  // the CTA-pair N = 128 halo kernel with the fp32 staged epilogue, no other epilogue term
  if (!(k.family == Family::kHalo && k.cg2 && !k.pair && k.block_n == 128 && p.y_f32 && k.staged && d->c_out % 128 == 0 &&
        !p.residual && p.sc_nch0 == 0 && !p.prelu_alpha && p.act == B200DM_ACT_NONE && p.post_act == B200DM_ACT_NONE)) {
    b200dm_set_error("conv_plan_set_fused_update: only on the CTA-pair fp32-output 3^3 conv with C_out %% 128 == 0");
    return B200DM_ERR_UNSUPPORTED;
  }
  B2_CHECK_ARG(u->sampler == 0 || u->sampler == 1, "conv_plan_set_fused_update: sampler must be 0 (ddpm) or 1 (ddim)");
  B2_CHECK_ARG(u->beta && u->sqrt_alpha && u->alpha_bar && u->alpha_bar_prev && u->sqrt_alpha_bar && u->sqrt_alpha_bar_prev &&
                   u->sqrt_one_minus_alpha_bar, "conv_plan_set_fused_update: null schedule table");
  B2_CHECK_ARG(u->batch == d->batch && u->n_per_sample == (int64_t)d->in_d * d->in_h * d->in_w * d->c_out,
               "conv_plan_set_fused_update: update geometry (%d x %lld) differs from the conv output", u->batch, (long long)u->n_per_sample);
  B2_CHECK_ARG((u->n_per_sample >> 2) < (1ll << 32), "conv_plan_set_fused_update: sample too large for the 32-bit Philox counter");
  B2_CHECK_ARG(x_t == x_prev, "conv_plan_set_fused_update: x_prev must alias x_t (the tile is updated in place through one tensor map)");
  B2_CHECK_ARG(((uintptr_t)x_t & 15) == 0 && ((uintptr_t)x_prev & 15) == 0 && ((uintptr_t)x_prev_16 & 15) == 0,
               "conv_plan_set_fused_update: pointers must be 16-byte aligned");
  EncodeTiledFn enc = b2_encode_tiled_fn();
  if (!enc) { b200dm_set_error("conv_plan_set_fused_update: cuTensorMapEncodeTiled unavailable"); return B200DM_ERR_CUDA; }
  const cuuint32_t box[5] = {16, 8, 16, 1, 1};   // one round of the fused epilogue: 16 columns x one 8 x 16 plane tile
  CUtensorMap my, mz;
  int rc = encode_act(enc, &my, "fused update x", x_prev, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d->c_out, d->in_w, d->in_h, d->in_d,
                      d->batch, box, CU_TENSOR_MAP_SWIZZLE_64B);
  if (!rc) rc = encode_act(enc, &mz, "fused update x16", x_prev_16, kTmapAct16, d->c_out, d->in_w, d->in_h, d->in_d, d->batch, box,
                           CU_TENSOR_MAP_SWIZZLE_32B);
  Variant fused = pl->v;
  fused.key.fuse = true;
  fused.key.ns = kHaloNSFused;
  if (!rc) rc = bind_kernel(pl, fused);
  if (rc) return rc;
  pl->om.y[0] = my; pl->om.y[1] = mz;
  pl->p.upd = *u; pl->p.upd_x = x_t;
  return B200DM_OK;
}

extern "C" int b200dm_conv_plan_set_shortcut(b200dm_conv_plan* pl, int32_t c0, int32_t c1, const void* x0, const void* x1,
                                             const void* w_packed, const float* bias) {
  B2_CHECK_ARG(pl && x0 && w_packed, "conv_plan_set_shortcut: null argument");
  const b200dm_conv_desc* d = &pl->desc;
  const KernelKey& k = pl->v.key;
  // the halo-reuse 3^3 kernel carries the segment as a runtime option of every instantiation: the plan keeps its kernel
  if (k.family != Family::kHalo || k.fuse) {
    b200dm_set_error("conv_plan_set_shortcut: only on plans of the 3^3 halo-reuse kernel without the fused update");
    return B200DM_ERR_UNSUPPORTED;
  }
  B2_CHECK_ARG(pl->p.sc_nch0 == 0, "conv_plan_set_shortcut: the plan already has a shortcut");
  B2_CHECK_ARG(c0 > 0 && c0 % 8 == 0 && c1 >= 0 && c1 % 8 == 0, "conv_plan_set_shortcut: C_in segments must be multiples of 8 (got %d,%d)", c0, c1);
  B2_CHECK_ARG((c1 > 0) == (x1 != nullptr), "conv_plan_set_shortcut: x1 must be given iff c1 > 0");
  B2_CHECK_ARG(((uintptr_t)x0 & 15) == 0 && ((uintptr_t)x1 & 15) == 0 && ((uintptr_t)w_packed & 15) == 0,
               "conv_plan_set_shortcut: pointers must be 16-byte aligned");
  EncodeTiledFn enc = b2_encode_tiled_fn();
  if (!enc) { b200dm_set_error("conv_plan_set_shortcut: cuTensorMapEncodeTiled unavailable"); return B200DM_ERR_CUDA; }
  const int nch0 = (c0 + 63) / 64, nch1 = (c1 + 63) / 64;
  const size_t ktot = pl->g.ktot + (size_t)(nch0 + nch1 + 2) / 3 * 3 * 64;   // + the shortcut's k-blocks, padded to whole 3-tap stages
  // the 3^3 segments' halo slab box: the kernel reads the shortcut at its centre tap
  const cuuint32_t box[5] = {64, 10, (cuuint32_t)(k.pair ? 2 : 18), (cuuint32_t)(k.pair ? 10 : 1), 1};
  CUtensorMap m0, m1, mb;
  int rc = encode_act(enc, &m0, "shortcut X", x0, kTmapAct16, c0, d->in_w, d->in_h, d->in_d, d->batch, box, CU_TENSOR_MAP_SWIZZLE_128B, 1,
                      1, k.pair);
  if (!rc) rc = encode_act(enc, &m1, "shortcut X", c1 > 0 ? x1 : x0, kTmapAct16, c1 > 0 ? c1 : c0, d->in_w, d->in_h, d->in_d, d->batch,
                           box, CU_TENSOR_MAP_SWIZZLE_128B, 1, 1, k.pair);
  if (!rc) rc = encode_weights3(enc, &mb, w_packed, pl->g, pl->v.wbox, ktot);
  if (rc) return rc;
  pl->mapSc0 = m0; pl->mapSc1 = m1; pl->mapB = mb;
  ConvParams& p = pl->p;
  p.sc_nch0 = nch0; p.sc_nch1 = nch1;
  p.sc_ksteps0_last = ((c0 - (nch0 - 1) * 64) + 15) / 16;
  p.sc_ksteps1_last = c1 > 0 ? ((c1 - (nch1 - 1) * 64) + 15) / 16 : 4;
  p.bias = bias;
  pl->flops += 2.0 * (c0 + c1) * d->c_out * (double)d->batch * pl->g.out_d * pl->g.out_h * pl->g.out_w;
  return B200DM_OK;
}

extern "C" int b200dm_conv_plan_info(const b200dm_conv_plan* p, int32_t* halo, int32_t* block_n, int32_t* ksplit) {
  B2_CHECK_ARG(p, "conv_plan_info: null plan");
  const Family f = p->v.key.family;
  if (halo) *halo = f == Family::kStencil ? 2 : (f == Family::kSweep ? 3 : (f != Family::kGemm ? 1 : 0));   // 2 = HBM-bound stencil-reduce kernel (C_out = 1), 3 = d-sweeping N = 96 kernel
  if (block_n) *block_n = p->v.key.block_n ? p->v.key.block_n : p->g.block_n;   // (stencil, sweep: the geometry's N tile)
  if (ksplit) *ksplit = p->p.ksplit;
  return B200DM_OK;
}

extern "C" int b200dm_conv_plan_set_out_affine(b200dm_conv_plan* p, const float* scale, const float* shift) {
  B2_CHECK_ARG(p, "conv_plan_set_out_affine: null plan");
  B2_CHECK_ARG((scale == nullptr) == (shift == nullptr), "conv_plan_set_out_affine: give both scale and shift, or neither");
  B2_CHECK_ARG(!scale || !p->p.prelu_alpha, "conv_plan_set_out_affine: not combinable with PReLU");
  B2_CHECK_ARG(!scale || !p->p.swap_ab, "conv_plan_set_out_affine: not combinable with a transposed store");
  B2_CHECK_ARG(!scale || p->v.key.family != Family::kStencil, "conv_plan_set_out_affine: not available on the C_out = 1 stencil plan");
  p->p.out_scale = scale;
  p->p.out_shift = shift;
  return B200DM_OK;
}

// GroupNorm statistics as a by-product of the producing conv (d-sweeping kernel only): the epilogue accumulates per-(item, channel)
// partial sums of the STORED values into `workspace` (double [rows][C][2], rows = batch * rows_per_sample); b200dm_gn_finalize
// turns them into (mean, rstd) in a fixed order.  Returns the workspace size, 0 when the plan cannot produce partials.
extern "C" size_t b200dm_conv_plan_gn_partials_bytes(const b200dm_conv_plan* p, int32_t* rows_per_sample) {
  if (!p || p->v.key.family != Family::kSweep) return 0;
  if (rows_per_sample) *rows_per_sample = p->wp.items / p->wp.batch * 2;
  return (size_t)p->wp.items * 2 * 32 * 2 * sizeof(double);
}

extern "C" int b200dm_conv_plan_set_gn_partials(b200dm_conv_plan* p, double* workspace, size_t ws_bytes) {
  B2_CHECK_ARG(p && workspace, "conv_plan_set_gn_partials: null argument");
  B2_CHECK_ARG(((uintptr_t)workspace & 7) == 0, "conv_plan_set_gn_partials: workspace must be 8-byte aligned");
  const size_t need = b200dm_conv_plan_gn_partials_bytes(p, nullptr);
  if (need == 0) { b200dm_set_error("conv_plan_set_gn_partials: this plan cannot produce GroupNorm partial sums"); return B200DM_ERR_UNSUPPORTED; }
  B2_CHECK_ARG(ws_bytes >= need, "conv_plan_set_gn_partials: workspace too small (%zu < %zu)", ws_bytes, need);
  p->wp.gn_part = workspace;
  return B200DM_OK;
}

int bind_gn_finalize(const double* partials, int32_t batch, int32_t rows_per_sample, int32_t c, int32_t groups,
                     int64_t voxels_per_sample, float eps, float* mean_rstd, BoundOp* op) {
  B2_CHECK_ARG(partials && mean_rstd && batch > 0 && rows_per_sample > 0 && c > 0 && groups > 0 && c % groups == 0 && voxels_per_sample > 0,
               "gn_finalize: bad argument");
  const double count = (double)voxels_per_sample * (c / groups);
  bind_launch(op, sweep::gn_finalize_kernel, dim3((unsigned)(batch * groups)), dim3(128), 0, partials, rows_per_sample, 1, c, groups, count, eps,
                  mean_rstd);
  return B200DM_OK;
}

extern "C" int b200dm_gn_finalize(const double* partials, int32_t batch, int32_t rows_per_sample, int32_t c, int32_t groups,
                                  int64_t voxels_per_sample, float eps, float* mean_rstd, void* stream) {
  return bind_and_run(bind_gn_finalize, stream, partials, batch, rows_per_sample, c, groups, voxels_per_sample, eps, mean_rstd);
}
