// 3^3 stride-1 'same' Conv3D with C_in = C_out = 32: d-SWEEPING persistent kernel (the decoders' 32 -> 32 convolutions at
// 128^3 / 64^3: vqgan_attn_cp.py:250-276 residual units, vqvae3d_monai.py:218-234).
//
// Why a second kernel.  At N = 32 the halo kernel (conv_halo.cuh) is bound by the shared-memory reads of the A operand: every
// M128 x N32 x K16 MMA re-reads 4 KB of the slab for 1 KB of weights, 27 taps x 2 planes -> 60-70 cycles per MMA against a
// 23-cycle tensor-pipe cost (profiles/r1h_ncu_halo32_staged.txt: tensor pipe 22 %, 26.6 GB crossing L2 -> SM for 4.3 GB of
// algorithmic traffic because the 64-channel chunk is half zero fill and the 27-tap weight set is re-streamed per tile).  Here:
//   * the three kd taps that read the SAME input plane are ONE N = 96 MMA: input plane p feeds output planes p+1 / p / p-1
//     (kd = 0 / 1 / 2), whose accumulators sit in three ADJACENT 32-column TMEM slots, so the A operand is read once instead
//     of three times (18 MMAs per plane instead of 54);
//   * a CTA walks one 8 w x 16 h column through all planes of its d range: every slab (10 x 18 voxels x 32 channels =
//     64-byte rows, SWIZZLE_64B -- no zero half) is loaded exactly once, there is no halo in d;
//   * the whole 27-tap weight set (54 KB as [kh,kw][kd][co][ci]) is loaded once per CTA and stays in shared memory.
// TMEM is a ring of R slots of 32 columns: plane G (a running index over the CTA's planes) owns slot R-1 - G % R, so the
// window {p+1, p, p-1} is ascending and contiguous except when it wraps (2 of R planes: two MMAs then).  A plane's first
// contribution (kd = 0, tap 0, k-step 0) is issued with accumulate = 0 on its own, so no slot is ever zeroed by hand.
//
// Warps (640 threads): 0 slab producer, 1 weight loader, 2 TMEM owner + MMA issuer, 3 idle (the epilogue warps must start at 4:
// TMEM lane quarter = warp % 4), 4-11 / 12-19 two epilogue groups that take alternate planes (an epilogue pass is ~1.5 k cycles of
// latency, the MMAs of a plane ~1.0 k).
// Input planes are staged and issued in PAIRS (one TMA box of two planes): the issuing thread's per-iteration bookkeeping
// (barrier waits, commits, index arithmetic: ~600 cycles, not overlapped because the tcgen05 queue is shallow) is paid once per two planes.
#pragma once
#include "conv_common.cuh"

namespace sweep {

constexpr int kThreads = 640;               // 20 warps
constexpr int kC = 32;
constexpr int kPlaneBytes = 180 * 64;       // one input plane of the column: 10 x 18 voxels x 64 B
constexpr int kSlabTx = 2 * kPlaneBytes;    // a slab = TWO consecutive input planes (one TMA box {32, 10, 18, 2, 1}): one barrier round
constexpr int kSlabBytes = 23 * 1024;       //          trip, one commit and one pass through the issuer's bookkeeping per two planes
constexpr int kNS = 3;                      // slab ring
constexpr int kR = 16;                      // TMEM ring: 16 slots x 32 columns = 512 columns
constexpr int kWBytes = 27 * 2048;          // [kh*3+kw][kd][32 co][32 ci] bf16, one 2 KB SWIZZLE_64B tile per tap
constexpr int kStgBytes = 8192;             // one plane tile: 128 rows x 64 B
constexpr size_t kSmem = 1024 + (size_t)kNS * kSlabBytes + kWBytes + 4 * kStgBytes + (2 * kNS + 1 + 2 * kR + 2) * 8 + 8 + 2 * 32 * 4 +
                         2 * 4 * 2 * 32 * 4 + 2 * 32 * 4;

struct Params {
  int D, H, W, batch;
  int tiles_w, tiles_h, dsplit, dlen, items;
  double* gn_part;   // optional [items][2 groups][32 channels][2] partial (sum, sum of squares) of the STORED values, else null
};

struct Item { int n, h0, w0, d0, d1; };
__device__ __forceinline__ Item decode(const Params& q, int item) {
  Item it;
  int r = item;
  const int ds = r % q.dsplit; r /= q.dsplit;
  const int tw = r % q.tiles_w; r /= q.tiles_w;
  const int th = r % q.tiles_h; r /= q.tiles_h;
  it.n = r; it.h0 = th * 16; it.w0 = tw * 8;
  it.d0 = ds * q.dlen; it.d1 = min(q.D, it.d0 + q.dlen);
  return it;
}

__device__ __forceinline__ void group_bar_sync(int g) { asm volatile("bar.sync %0, 256;" ::"r"(g + 1) : "memory"); }

constexpr uint64_t kLayoutSw64 = 4;

constexpr uint32_t kIdesc32 = ptx::make_idesc_act(128, 32), kIdesc64 = ptx::make_idesc_act(128, 64), kIdesc96 = ptx::make_idesc_act(128, 96);
__host__ __device__ constexpr uint32_t idesc_of(int nkd) { return nkd == 1 ? kIdesc32 : (nkd == 2 ? kIdesc64 : kIdesc96); }

// One MMA group over the kd range [A, B] whose first N1 slots fit before the ring wraps (N1 >= B - A + 1: no wrap).
template <int A, int B, int N1>
__device__ __forceinline__ void mma_range(uint32_t tmem_base, uint32_t s0, uint64_t da, uint64_t db, uint32_t acc) {
  constexpr int n = B - A + 1;
  if constexpr (n > 0) {
    const uint32_t col = tmem_base + 32 * ((s0 + A) & (kR - 1));
    if constexpr (N1 >= n || N1 <= 0) {   // (N1 <= 0: the whole range lies after the wrap; col is already the wrapped slot)
      ptx::tc_mma_f16(col, da, db + (uint64_t)(A * (2048 >> 4)), idesc_of(n), acc);
    } else {
      ptx::tc_mma_f16(col, da, db + (uint64_t)(A * (2048 >> 4)), idesc_of(N1), acc);
      ptx::tc_mma_f16(tmem_base, da, db + (uint64_t)((A + N1) * (2048 >> 4)), idesc_of(n - N1), acc);
    }
  }
}

// All MMAs of one input plane: kd range [KLO, KHI]; N1 = how many of those slots (counted from KLO) lie before the ring wrap.
// Fully unrolled: every operand offset is an immediate, the single issuing thread spends ~5 integer instructions per MMA
// (a generic loop with run-time segments issued one MMA per ~135 cycles against ~56 cycles of execution).
template <int KLO, int KHI, int N1>
__device__ __forceinline__ void issue_plane(uint32_t tmem_base, uint32_t s0, uint64_t a_pl, uint64_t b_desc0) {
#pragma unroll
  for (int k9 = 0; k9 < 9; ++k9) {
    const uint64_t da = a_pl + (uint64_t)(((k9 / 3) * 10 + (k9 % 3)) * 4);   // (kh*10 + kw) rows of 64 B in 16-byte units
    const uint64_t db = b_desc0 + (uint64_t)(k9 * 3 * (2048 >> 4));
    if (k9 == 0 && KLO == 0) {
      // the plane opened by this input plane (kd = 0): its first contribution overwrites the slot
      ptx::tc_mma_f16(tmem_base + 32 * s0, da, db, kIdesc32, 0u);
      mma_range<1, KHI, N1 - 1>(tmem_base, s0, da, db, 1u);
    } else {
      mma_range<KLO, KHI, N1>(tmem_base, s0, da, db, 1u);
    }
    mma_range<KLO, KHI, N1>(tmem_base, s0, da + 2, db + 2, 1u);   // channels 16..31: +32 B on both operands
  }
}

__global__ void __launch_bounds__(kThreads, 1)
conv_sweep32_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapW,
                    const __grid_constant__ CUtensorMap mapY, const __grid_constant__ CUtensorMap mapR, const ConvParams p, const Params q) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_s = smem + kNS * kSlabBytes;
  uint8_t* stg_base = w_s + kWBytes;                     // [group][2 buffers][8 KB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg_base + 4 * kStgBytes);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * kNS + 1 + 2 * kR + 2);
  float* bias_s = reinterpret_cast<float*>(tmem_ptr_smem + 2);   // [bias | scale][32] (16-byte aligned)
  float* red_s = bias_s + 64;                                     // [group][quarter][half][16 columns][2]
  float* piv_s = red_s + 2 * 4 * 2 * 32;                          // [group][32 channels]: GroupNorm pivots of the current item

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t slab_base = ptx::smem_u32(smem), w_base = ptx::smem_u32(w_s), bar_base = ptx::smem_u32(bars);
  auto slab_full = [&](int s) { return bar_base + 8u * s; };
  auto slab_empty = [&](int s) { return bar_base + 8u * (kNS + s); };
  const uint32_t w_full = bar_base + 8u * (2 * kNS);
  auto acc_full = [&](int s) { return bar_base + 8u * (2 * kNS + 1 + s); };
  auto acc_empty = [&](int s) { return bar_base + 8u * (2 * kNS + 1 + kR + s); };
  auto res_bar = [&](int g) { return bar_base + 8u * (2 * kNS + 1 + 2 * kR + g); };   // residual tile of epilogue group g has landed

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int s = 0; s < kNS; ++s) { ptx::mbar_init(slab_full(s), 1); ptx::mbar_init(slab_empty(s), 1); }
    ptx::mbar_init(w_full, 1);
    for (int s = 0; s < kR; ++s) { ptx::mbar_init(acc_full(s), 1); ptx::mbar_init(acc_empty(s), 8); }
    ptx::mbar_init(res_bar(0), 1); ptx::mbar_init(res_bar(1), 1);
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&mapX);
    ptx::prefetch_tmap(&mapW);
    ptx::prefetch_tmap(&mapY);
    if (p.residual) ptx::prefetch_tmap(&mapR);
  }
  if (warp == 2) { ptx::tmem_alloc(ptx::smem_u32(tmem_ptr_smem), 32 * kR); ptx::tmem_relinquish(); }
  if (threadIdx.x >= 128 && threadIdx.x < 128 + 32) {   // bias / output affine of the 32 channels: constant for the whole launch
    const int c = threadIdx.x - 128;
    float b = p.bias ? __ldg(p.bias + c) : 0.f, sc = 1.f;
    if (p.out_scale) { sc = __ldg(p.out_scale + c); b = fmaf(sc, b, __ldg(p.out_shift + c)); }
    bias_s[c] = b; bias_s[32 + c] = sc;
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();

  if (warp == 0) {
    // ===================== slab producer: one box per input plane of the column =====================
    uint32_t s = 0, ph = 1;
    int tis = 0;
    bool ok = true;
    for (int item = blockIdx.x; item < q.items && ok; item += gridDim.x) {
      const Item it = decode(q, item);
      for (int pl = it.d0 - 1; pl <= it.d1 && ok; pl += 2) {   // (an odd count loads one plane past the range: never used)
        ok = ptx::mbar_wait_sleep(slab_empty(s), ph, p.dbg, 0x5301);
        if (!ok) break;
        if (lane == 0) trace_ev(p, 2, tis, 20);
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(slab_full(s), kSlabTx);
          ptx::tma_load_5d(slab_base + s * kSlabBytes, &mapX, slab_full(s), 0, it.w0 - 1, it.h0 - 1, pl, it.n);
        }
        __syncwarp();
        if (++s == kNS) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== weights: 27 tiles of [32 co][32 ci], resident for the whole launch =====================
    if (ptx::elect_one()) {
      ptx::mbar_expect_tx(w_full, kWBytes);
      for (int kd = 0; kd < 3; ++kd)
        for (int k9 = 0; k9 < 9; ++k9) ptx::tma_load_3d(w_base + (k9 * 3 + kd) * 2048, &mapW, w_full, 0, 0, kd * 9 + k9);
    }
    __syncwarp();
  } else if (warp == 2) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      bool ok = ptx::mbar_wait(w_full, 0, p.dbg, 0x5302);
      const uint64_t a_desc0 = ptx::make_smem_desc(slab_base, 16, 640, kLayoutSw64);   // 8-row groups 10 rows (640 B) apart
      const uint64_t b_desc0 = ptx::make_smem_desc(w_base, 16, 512, kLayoutSw64);
      uint32_t s = 0, ph = 0;
      int ti = 0;
      uint32_t gbase = 0;     // running plane index of the item's first output plane
      uint32_t drained = 0;   // every plane with running index < drained is known to have left TMEM
      // all MMAs of input plane pi of the current column (kd range by position, ring wrap by slot) + the commit of the output plane
      // that received its last contribution
      auto plane = [&](int pi, int nout, uint64_t a_pl) {
        const int kd_lo = pi - nout + 1 > 0 ? pi - nout + 1 : 0, kd_hi = pi < 2 ? pi : 2;
        const uint32_t G0 = gbase + (uint32_t)pi;               // running index of the plane this input plane opens (kd = 0)
        const uint32_t s0 = (kR - 1) - (G0 & (kR - 1));         // its TMEM slot; kd = 1, 2 -> slots s0 + 1, s0 + 2 (mod R)
        if (kd_lo == 0 && kd_hi == 2 && s0 <= (uint32_t)(kR - 3)) {
          issue_plane<0, 2, 3>(tmem_base, s0, a_pl, b_desc0);   // interior plane, window not wrapping: all but ~2 of R + 4 per column
        } else {
          const uint32_t sa = (s0 + (uint32_t)kd_lo) & (kR - 1), nkd = (uint32_t)(kd_hi - kd_lo + 1);
          const uint32_t n1 = nkd < kR - sa ? nkd : kR - sa;    // slots of the window before the ring wraps
          switch (kd_lo * 16 + kd_hi * 4 + (int)n1) {
            case 0 * 16 + 2 * 4 + 2: issue_plane<0, 2, 2>(tmem_base, s0, a_pl, b_desc0); break;
            case 0 * 16 + 2 * 4 + 1: issue_plane<0, 2, 1>(tmem_base, s0, a_pl, b_desc0); break;
            case 0 * 16 + 1 * 4 + 2: issue_plane<0, 1, 2>(tmem_base, s0, a_pl, b_desc0); break;   // second input plane of a column
            case 0 * 16 + 1 * 4 + 1: issue_plane<0, 1, 1>(tmem_base, s0, a_pl, b_desc0); break;
            case 0 * 16 + 0 * 4 + 1: issue_plane<0, 0, 1>(tmem_base, s0, a_pl, b_desc0); break;   // first input plane (d0 - 1)
            case 1 * 16 + 2 * 4 + 2: issue_plane<1, 2, 2>(tmem_base, s0, a_pl, b_desc0); break;   // input plane d1 - 1
            case 1 * 16 + 2 * 4 + 1: issue_plane<1, 2, 1>(tmem_base, s0, a_pl, b_desc0); break;
            case 2 * 16 + 2 * 4 + 1: issue_plane<2, 2, 1>(tmem_base, s0, a_pl, b_desc0); break;   // last input plane (d1)
            case 1 * 16 + 1 * 4 + 1: issue_plane<1, 1, 1>(tmem_base, s0, a_pl, b_desc0); break;   // one-plane columns
            default: if (p.dbg) atomicExch(p.dbg, 0x53ff); break;
          }
        }
        if (kd_hi == 2) ptx::tc_commit(acc_full((s0 + 2) & (kR - 1)));   // output plane d0 + pi - 2 is complete
      };
      for (int item = blockIdx.x; item < q.items && ok; item += gridDim.x) {
        const Item it = decode(q, item);
        const int nout = it.d1 - it.d0;
        for (int pi = 0; pi < nout + 2 && ok; pi += 2) {
          // Slot reuse: before plane G is opened, plane G - R must have been drained.  The two epilogue groups drain their planes
          // in order, so ONE check of the two newest complete planes (both parities) every 8 planes covers the next 8 openings
          // instead of an mbarrier round trip (~110 cycles on this thread) per plane.
          const uint32_t Gn = gbase + (uint32_t)(pi + 1 < nout ? pi + 1 : nout - 1);   // newest plane this pair opens
          if (pi < nout && drained + (kR - 1) < Gn) {
            const uint32_t T = Gn - 7;   // planes T-1, T-2 are complete (their last contribution came at least 4 input planes ago)
            trace_ev(p, 0, ti, 1);
            for (uint32_t j = T - 2; j < T && ok; ++j)
              ok = ptx::mbar_wait(acc_empty((kR - 1) - (j & (kR - 1))), (j / kR) & 1, p.dbg, 0x5303);
            if (!ok) break;
            drained = T;
            trace_ev(p, 0, ti, 2);
          }
          ok = ptx::mbar_wait(slab_full(s), ph, p.dbg, 0x5304);
          if (!ok) break;
          trace_ev(p, 0, ti, 3);
          ptx::tc_fence_after();
          const uint64_t a_pl = a_desc0 + (uint64_t)(s * (uint32_t)(kSlabBytes >> 4));
          plane(pi, nout, a_pl);
          if (pi + 1 < nout + 2) plane(pi + 1, nout, a_pl + (uint64_t)(kPlaneBytes >> 4));
          ptx::tc_commit(slab_empty(s));
          trace_ev(p, 0, ti, 4);
          if (++s == kNS) { s = 0; ph ^= 1; }
        }
        gbase += (uint32_t)nout;
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 20) {
    // ===================== epilogue: group e = (warp - 4) / 8 takes the planes with running index G % 2 == e =====================
    const int e = (warp - 4) >> 3, wg = (warp - 4) & 7;
    const int qd = warp & 3, half = wg >> 2;
    const int r = qd * 32 + lane, iw = r & 7, ih = r >> 3;
    const int gtid = threadIdx.x - 128 - e * 256;
    uint8_t* stg_g = stg_base + e * 2 * kStgBytes;
    const float* bs = bias_s + 16 * half;
    const float* scs = p.out_scale ? bias_s + 32 + 16 * half : nullptr;
    uint32_t gbase = 0, nstore = 0;
    int ti = 0;
    const bool trw = warp == 4 && lane == 0;
    bool ok = true;
    for (int item = blockIdx.x; item < q.items && ok; item += gridDim.x) {
      const Item it = decode(q, item);
      const int nout = it.d1 - it.d0;
      const int ow = it.w0 + iw, oh = it.h0 + ih;
      const bool inb = ow < q.W && oh < q.H;
      float sacc = 0.f;   // GroupNorm partial of (channel, statistic) pair `lane` over this warp's rows and planes (see below)
      bool first = true;  // this group's first plane of the item: its row 0 (always inside the volume) gives the pivots
      for (int pq = 0; pq < nout && ok; ++pq) {
        const uint32_t G = gbase + (uint32_t)pq;
        if ((int)(G & 1) != e) continue;
        const int od = it.d0 + pq;
        const uint32_t sl = kR - 1 - G % kR;
        // residual tile (the output tile's own box) -> TMA-loaded INTO this plane's staging buffer while the accumulator is
        // still in flight; each thread later reads its 32 bytes from the chunks it overwrites with the result.  (Row-per-thread
        // global loads of the residual cost the LSU ~16 lines per instruction: the conv2 launches ran 2.44 ms against 1.81 ms
        // for the same conv without a residual.)
        const bool res = p.residual != nullptr;
        uint8_t* stg = stg_g + (nstore & 1) * kStgBytes;
        if (res && gtid == 0) {
          ptx::bulk_wait_read_1();   // the store that last used this buffer has finished reading it
          ptx::mbar_expect_tx(res_bar(e), kStgBytes);
          ptx::tma_load_5d(ptx::smem_u32(stg), &mapR, res_bar(e), 0, it.w0, it.h0, od, it.n);
        }
        if (trw) trace_ev(p, 1, ti, 10);
        ok = ptx::mbar_wait_sleep(acc_full(sl), (G / kR) & 1, p.dbg, 0x5305);
        if (!ok) break;
        if (trw) trace_ev(p, 1, ti, 11);
        ptx::tc_fence_after();
        uint32_t ra[16];
        ptx::tc_ld_32x32b_x16(tmem_base + ((uint32_t)(qd * 32) << 16) + 32 * sl + 16 * half, ra);
        ptx::tc_wait_ld();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(acc_empty(sl));   // the slot may be re-opened while this plane is stored
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(ra[j]);
        if (scs) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] *= scs[j];
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] += bs[j];
        if (p.act != B200DM_ACT_NONE) {
          apply_act_vec(v, p.act);
        }
        const int ch = 2 * half, sw = (r >> 1) & 3;   // 64-byte rows, SWIZZLE_64B: 16-byte chunk ^= (row / 2) % 4
        if (res) {
          ok = ptx::mbar_wait_sleep(res_bar(e), nstore & 1, p.dbg, 0x5306, 32);
          if (!ok) break;
          float a[16];
          unpack8(*reinterpret_cast<const bf16x8*>(stg + r * 64 + (((ch) ^ sw) << 4)), *reinterpret_cast<float(*)[8]>(&a[0]));
          unpack8(*reinterpret_cast<const bf16x8*>(stg + r * 64 + (((ch + 1) ^ sw) << 4)), *reinterpret_cast<float(*)[8]>(&a[8]));
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] += a[j];
        }
        if (p.post_act != B200DM_ACT_NONE) {
          apply_act_vec(v, p.post_act);
        }
        const bf16x8 o0 = pack8(*reinterpret_cast<float(*)[8]>(&v[0])), o1 = pack8(*reinterpret_cast<float(*)[8]>(&v[8]));
        if (q.gn_part && first && r == 0) {
          float w[16];
          unpack8(o0, *reinterpret_cast<float(*)[8]>(&w[0]));
          unpack8(o1, *reinterpret_cast<float(*)[8]>(&w[8]));
#pragma unroll
          for (int j = 0; j < 16; ++j) piv_s[e * 32 + 16 * half + j] = w[j];   // read after the group barrier below
        }
        first = false;
        if (!res) {   // (with a residual the buffer was claimed before its tile was loaded, and every thread has seen that load land)
          if (gtid == 0) ptx::bulk_wait_read_1();   // the store that last used this buffer has finished reading it
          group_bar_sync(e);
        }
        *reinterpret_cast<bf16x8*>(stg + r * 64 + (((ch) ^ sw) << 4)) = o0;
        *reinterpret_cast<bf16x8*>(stg + r * 64 + (((ch + 1) ^ sw) << 4)) = o1;
        ptx::fence_proxy_async();
        group_bar_sync(e);
        if (gtid == 0) {
          ptx::tma_store_5d(&mapY, ptx::smem_u32(stg), 0, it.w0, it.h0, od, it.n);
          ptx::bulk_commit_group();
        }
        if (q.gn_part) {
          // GroupNorm statistics of the tensor as STORED (rounded), as sums of d = y - K[channel] (pivots of this item, so the fp32
          // sums do not carry the channel's offset: see gn_partial_kernel).  32 values per row (16 sums, 16 squares) are reduce-SCATTERED
          // over the warp's 32 rows: after 5 exchange steps (16 + 8 + 4 + 2 + 1 shuffles) lane L holds the total of value L, so the
          // running sums take ONE register per thread instead of 32 (640 threads share the register file).
          float w[32];
          unpack8(o0, *reinterpret_cast<float(*)[8]>(&w[0]));
          unpack8(o1, *reinterpret_cast<float(*)[8]>(&w[8]));
          const float* pv = piv_s + e * 32 + 16 * half;
#pragma unroll
          for (int j = 0; j < 16; ++j) { w[j] = inb ? w[j] - pv[j] : 0.f; w[16 + j] = w[j] * w[j]; }
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) {
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int j = 0; j < o; ++j) {
              const float send = up ? w[j] : w[j + o], keep = up ? w[j + o] : w[j];
              w[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
          }
          sacc += w[0];
        }
        if (trw) trace_ev(p, 1, ti, 12);
        ++nstore;
      }
      if (q.gn_part) {
        // column sums of this group's planes: 4 lane quarters -> shared memory -> one value per (channel, statistic), fixed order
        red_s[((e * 4 + qd) * 2 + half) * 32 + lane] = sacc;   // lane < 16: sum of channel 16*half + lane; else sum of squares
        group_bar_sync(e);
        if (gtid < 64) {   // (channel, stat) pair gtid: channel = gtid / 2; fp64 (sum, sum of squares) of y rebuilt from the pivot
          const int c = gtid >> 1, st = gtid & 1, hf = c >> 4, cj = c & 15;
          float s1 = 0.f, s2 = 0.f;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            s1 += red_s[((e * 4 + k) * 2 + hf) * 32 + cj];
            s2 += red_s[((e * 4 + k) * 2 + hf) * 32 + cj + 16];
          }
          const int f = (e - (int)gbase) & 1;                      // this group's first plane of the item
          const int planes = nout > f ? (nout - f + 1) >> 1 : 0;
          const double cnt = (double)planes * min(8, q.W - it.w0) * min(16, q.H - it.h0);
          const double K = planes ? (double)piv_s[e * 32 + c] : 0.0;
          q.gn_part[(((size_t)item * 2 + e) * 32 + c) * 2 + st] =
              st ? cnt * K * K + 2.0 * K * (double)s1 + (double)s2 : cnt * K + (double)s1;
        }
        group_bar_sync(e);
      }
      gbase += (uint32_t)nout;
    }
    if (gtid == 0) ptx::bulk_wait_read_all();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) { ptx::tc_fence_after(); ptx::tmem_dealloc(tmem_base, 32 * kR); }
}

// mean / rstd of GroupNorm from the conv's per-item partial sums: one block per (sample, group), fixed summation order
// (items ascending, then channels) in double precision -> the chain stays bit-reproducible.
__global__ void __launch_bounds__(128) gn_finalize_kernel(const double* __restrict__ part, int items_per_sample, int parts, int C,
                                                          int groups, double count, float eps, float* __restrict__ mean_rstd) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = blockIdx.x / groups, g = blockIdx.x % groups, cpg = C / groups;
  __shared__ double s_sum[128], s_sq[128];
  double a = 0.0, b = 0.0;
  const int rows = items_per_sample * parts;
  for (int i = threadIdx.x; i < rows; i += 128) {
    const double* pr = part + (((size_t)n * rows + i) * C + (size_t)g * cpg) * 2;
    for (int c = 0; c < cpg; ++c) { a += pr[2 * c]; b += pr[2 * c + 1]; }
  }
  s_sum[threadIdx.x] = a; s_sq[threadIdx.x] = b;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) { s_sum[threadIdx.x] += s_sum[threadIdx.x + o]; s_sq[threadIdx.x] += s_sq[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double m = s_sum[0] / count;
    double var = s_sq[0] / count - m * m;
    if (var < 0.0) var = 0.0;
    mean_rstd[((size_t)n * groups + g) * 2] = (float)m;
    mean_rstd[((size_t)n * groups + g) * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
  }
}

}  // namespace sweep
