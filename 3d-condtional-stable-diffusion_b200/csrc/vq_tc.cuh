// K11 on the tensor cores, bit-identical indices.
//
// vq_kernel (vq.cu) evaluates all N x K distances with fp32 SIMT FMAs because the ranking has to be reproducible to the last bit
// (45 TFLOP/s: the FMA and shared-memory pipes are co-saturated).  Here the N x K products run on tcgen05 as a CANDIDATE search,
// and only the few codes that can possibly be the first minimum are re-evaluated with vq_kernel's exact fp32 chain:
//
//   split     x * 2^sx = x_hi + x_lo,  e * 2^se = e_hi + e_lo   (two IEEE fp16 terms each = 22 significand bits; sx per row from the row's
//             max, se per codebook, so nothing leaves the normal fp16 range; the products of fp16 values are exact in fp32)
//   scores    s~ = x_hi.e_hi + x_lo.e_hi + x_hi.e_lo            (three K = D passes of kind::f16 MMAs into one fp32 accumulator tile)
//   bound     |s~ / 2^(sx+se) - s| <= errS = 2 D 2^-24 ||x|| max||e||    (s = the exact chain's value: its own rounding error is
//             <= D 2^-24 sum|x_d e_d|, the dropped x_lo.e_lo term and the split remainders are < 2^-20, the MMA's fp32
//             accumulation over 3 D / 16 steps is budgeted the remaining D 2^-24)
//   candidates  every code with  g~_k = ||e_k||^2 - 2 s~_k  <=  min_k g~_k + M,   M = 2 (2 errS + U),  U = 2^-21 (||x||^2 + max||e||^2)
//             (U covers the roundings of fl(fl(||x||^2 + ||e||^2) - 2 s)); the exact first minimum is provably among them
//   recheck   one candidate: done.  Several (near-ties, ~1/3 of the rows at cfg-3): vq_kernel's chain -- ascending-d fp32 FMAs,
//             sequential ||x||^2, fl(fl(||x||^2 + ||e||^2) - 2 s), lowest index on ties -- for those codes only.
//   fallback  rows with a non-finite element or more candidates than the list holds: the full exact scan by the row's thread.
//
// CTA = 128 rows.  A = [x_hi | x_lo] (128 KB at D = 256) is built once in shared memory by all warps (coalesced fp32 loads, row
// scale by shuffles over the 8 lanes of a row, SWIZZLE_128B K-major stores); the codebook halves stream through a TMA ring of 16 KB tiles (128 codes x 64
// columns), each e_hi tile serving the x_hi and the x_lo pass; the score tile (128 x 128 fp32) is double-buffered in TMEM so the
// candidate scan of code tile j overlaps the MMAs of tile j + 1.
// Warps (384 threads): 0 = TMA producer, 1 = TMEM owner + MMA issuer, 4-11 = candidate scan (thread = row = TMEM lane; two warps per
// lane quarter, each takes one 64-column half of every score tile and keeps its own running minimum and candidate list; the lists
// are merged at the end by the warps of half 0, which also run the rechecks).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include "common.cuh"
#include "ptx.cuh"

namespace vqtc {

constexpr int kThreads = 384;   // 4 role warps + 8 scan warps
constexpr int kNSB = 4;        // codebook tile ring
constexpr int kTile = 16384;   // 128 rows x 128 B
constexpr int kCap = 10;       // candidates kept per (row, column half)

struct Params {
  int64_t n;
  int k, d;
  const void* x;
  int x_f32, q_f32;
  const float* cb;       // (K, D) fp32
  const float* esq;      // (K) exact sequential ||e||^2 (sqnorm_kernel)
  const float* meta;     // [0] = max ||e||^2, [1] = 2^-se, [2] = max |e|, [3] != 0: codebook outside the scaled range (full scans)
  int64_t* idx;
  void* q;
  int32_t* hist;
  int* dbg;
  int wave_ctas;         // CTAs resident at once (1 per SM): block b + wave_ctas runs on an SM after block b
  float margin_scale;    // 1 in production; tests shrink it to measure the headroom of the error bound
  unsigned long long* stats;   // optional [3]: rows rechecked, candidates rechecked, rows that fell back to the full scan
};

__host__ __device__ constexpr uint32_t idesc_f16(int m, int n) {   // kind::f16, A/B = IEEE fp16 (format 0), D = fp32, K-major both
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void scan_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 scan warps

template <bool kX16>
__device__ __forceinline__ float4 load_x4(const void* x, int64_t off) {   // 4 consecutive elements, off % 4 == 0
  if (kX16) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const act_t*>(x) + off));
    act2_t h[2];
    memcpy(h, &u, 8);
    const float2 a = act2_to_float2(h[0]), b = act2_to_float2(h[1]);
    return make_float4(a.x, a.y, b.x, b.y);
  }
  return __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + off));
}

// vq_kernel's exact distance of row `xr` to code k (same operations in the same order: bit-identical)
template <bool kX16>
__device__ __forceinline__ float exact_dist(const Params& p, int64_t row, int k, float xsq) {
  const float* e = p.cb + (int64_t)k * p.d;
  float acc = 0.f;
#pragma unroll 4
  for (int d = 0; d < p.d; d += 4) {
    const float4 ev = __ldg(reinterpret_cast<const float4*>(e + d));
    const float4 xv = load_x4<kX16>(p.x, row * p.d + d);
    acc = fmaf(xv.x, ev.x, acc);
    acc = fmaf(xv.y, ev.y, acc);
    acc = fmaf(xv.z, ev.z, acc);
    acc = fmaf(xv.w, ev.w, acc);
  }
  return __fsub_rn(__fadd_rn(xsq, __ldg(p.esq + k)), __fmul_rn(2.0f, acc));
}
template <bool kX16>
__device__ __forceinline__ float exact_xsq(const Params& p, int64_t row) {
  float s = 0.f;
#pragma unroll 4
  for (int d = 0; d < p.d; d += 4) {
    const float4 v = load_x4<kX16>(p.x, row * p.d + d);
    s = __fadd_rn(s, __fmul_rn(v.x, v.x));
    s = __fadd_rn(s, __fmul_rn(v.y, v.y));
    s = __fadd_rn(s, __fmul_rn(v.z, v.z));
    s = __fadd_rn(s, __fmul_rn(v.w, v.w));
  }
  return s;
}

// candidate list of one row (shared memory, ascending k): append (k, g); when full, first drop what the running minimum has left
// behind.  Returns the new count, or -1 when the list overflows (the row then takes the full exact scan).
__device__ __noinline__ int cand_push(int* ck, float* cg, int cnt, int k, float g, float thr) {
  if (cnt == kCap) {
    int w = 0;
    for (int i = 0; i < kCap; ++i)
      if (cg[i] <= thr) { ck[w] = ck[i]; cg[w] = cg[i]; ++w; }
    cnt = w;
    if (cnt == kCap) return -1;
  }
  ck[cnt] = k;
  cg[cnt] = g;
  return cnt + 1;
}

template <bool kX16>
__global__ void __launch_bounds__(kThreads, 1)
vq_tc_kernel(const __grid_constant__ CUtensorMap mapHi, const __grid_constant__ CUtensorMap mapLo, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
  const int DC = p.d >> 6;                                  // 64-column chunks of the K dimension
  uint8_t* a_hi = smem;                                     // [DC][128 rows][128 B]
  uint8_t* a_lo = a_hi + DC * kTile;
  uint8_t* b_ring = a_lo + DC * kTile;                      // [kNSB][128 codes][128 B]
  float* e2_s = reinterpret_cast<float*>(b_ring + kNSB * kTile);   // [K]
  float* inv_s = e2_s + p.k;                                // [128] 2^-(sx_r + se): score -> x.e
  float* marg_s = inv_s + 128;                              // [128] candidate margin M of the row (< 0: fallback row)
  int* cand_k = reinterpret_cast<int*>(marg_s + 128);       // [2 halves][128][kCap]
  float* cand_g = reinterpret_cast<float*>(cand_k + 256 * kCap);
  float* half_min = cand_g + 256 * kCap;                    // [2][128] running minimum of each half (overflow: -inf)
  int* half_cnt = reinterpret_cast<int*>(half_min + 256);   // [2][128]
  int* final_idx = half_cnt + 256;
  uint64_t* bars = reinterpret_cast<uint64_t*>(final_idx + 128);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * kNSB + 4);
  const uint32_t a_hi_base = ptx::smem_u32(a_hi), a_lo_base = ptx::smem_u32(a_lo), b_base = ptx::smem_u32(b_ring);
  const uint32_t bar_base = ptx::smem_u32(bars);
  auto b_full = [&](int s) { return bar_base + 8u * s; };
  auto b_empty = [&](int s) { return bar_base + 8u * (kNSB + s); };
  auto s_full = [&](int b) { return bar_base + 8u * (2 * kNSB + b); };
  auto s_free = [&](int b) { return bar_base + 8u * (2 * kNSB + 2 + b); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)blockIdx.x * 128;
  const int ntile = p.k >> 7;
  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int s = 0; s < kNSB; ++s) { ptx::mbar_init(b_full(s), 1); ptx::mbar_init(b_empty(s), 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(s_full(b), 1); ptx::mbar_init(s_free(b), 8); }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&mapHi);
    ptx::prefetch_tmap(&mapLo);
  }
  if (warp == 1) { ptx::tmem_alloc(ptx::smem_u32(tmem_ptr_smem), 256); ptx::tmem_relinquish(); }
  pdl_wait();
  const float e2max = __ldg(p.meta), se_inv = __ldg(p.meta + 1), emax = __ldg(p.meta + 2);
  const bool codebook_bad = __ldg(p.meta + 3) != 0.f;   // non-finite / out-of-range codebook: every row takes the full exact scan
  for (int i = threadIdx.x; i < p.k; i += kThreads) e2_s[i] = __ldg(p.esq + i);

  // ---- A operand: a warp converts 4 rows at a time (8 lanes per row, each lane 4 consecutive columns of every 32-column group: the
  // 8 lanes of a row read 128 contiguous bytes per load).  The 4 rows of a trip differ in bit 2 / bit 0 of the row number so that
  // their swizzled 64-byte store segments fall into different bank halves.  Loads of trip i + 1 are in flight during trip i.
  if (warp < 8) {
    const int sub = lane >> 3, ll = lane & 7;
    const int ngrp = p.d >> 5;   // 32-column groups (<= 8)
    auto row_of = [&](int it) { return warp * 16 + (it >> 1) * 8 + (it & 1) * 2 + (sub & 1) * 4 + (sub >> 1); };
    auto load_row = [&](int it, float4 (&v)[8]) {
      const int64_t row = row0 + row_of(it);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < ngrp && row < p.n) v[j] = load_x4<kX16>(p.x, row * p.d + j * 32 + ll * 4);
      }
    };
    float4 cur[8], nxt[8];
    load_row(0, cur);
#pragma unroll 1
    for (int it = 0; it < 4; ++it) {
      if (it + 1 < 4) load_row(it + 1, nxt);
      const int r = row_of(it);
      const int64_t row = row0 + r;
      float amax = 0.f, ssq = 0.f;
      bool bad = false;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float t[4] = {cur[j].x, cur[j].y, cur[j].z, cur[j].w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (!(fabsf(t[q]) <= 3.0e38f)) bad = true;   // NaN / inf
          amax = fmaxf(amax, fabsf(t[q]));
          ssq = fmaf(t[q], t[q], ssq);
        }
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {   // over the 8 lanes of the row
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
        ssq += __shfl_xor_sync(0xffffffffu, ssq, o);
        const int other_bad = __shfl_xor_sync(0xffffffffu, (int)bad, o);   // unconditional: every lane takes part in the shuffle
        bad = bad || other_bad != 0;
      }
      bad = bad || (amax != 0.f && !(amax >= 9.0e-13f && amax <= 1.0e12f)) || codebook_bad;   // scales stay well inside fp32
      // row scale 2^sx with max |x| 2^sx in [2^13, 2^14): fp16 hi / lo stay normal for every element within 2^-12 of the row's max
      int ex = 0;
      if (amax > 0.f) { (void)frexpf(amax, &ex); }
      const int sx = (amax > 0.f && !bad) ? 14 - ex : 0;
      const float sc = bad ? 0.f : ldexpf(1.0f, sx);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (j < ngrp) {
          const float t[4] = {cur[j].x, cur[j].y, cur[j].z, cur[j].w};
          __half h[4], l[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float ts = bad ? 0.f : t[q] * sc;                    // exact (power of two)
            h[q] = __float2half_rn(ts);
            l[q] = __float2half_rn(ts - __half2float(h[q]));           // exact difference, rounded to 11 bits
          }
          const int c = j * 32 + ll * 4, chunk = c >> 6, col = c & 63;
          const uint32_t off = (uint32_t)chunk * kTile + (uint32_t)r * 128u + ((((uint32_t)col >> 3) ^ ((uint32_t)r & 7u)) << 4) + (((uint32_t)col & 7u) << 1);
          uint2 hv, lv;
          memcpy(&hv, h, 8);
          memcpy(&lv, l, 8);
          *reinterpret_cast<uint2*>(a_hi + off) = hv;
          *reinterpret_cast<uint2*>(a_lo + off) = lv;
        }
      }
      if (ll == 0) {
        inv_s[r] = ldexpf(se_inv, -sx);
        const float xsq_ub = ssq * 1.001f, xn = sqrtf(xsq_ub), en = sqrtf(e2max);
        const float errS = 2.0f * (float)p.d * 5.9604645e-8f * xn * en + 1.0e-30f + 3.0e-10f * emax * xn * sqrtf((float)p.d);
        const float U = 4.7683716e-7f * (xsq_ub + e2max);
        marg_s[r] = (bad || row >= p.n) ? -1.0f : p.margin_scale * 2.0f * (2.0f * errS + U);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) cur[j] = nxt[j];
    }
  }
  ptx::fence_proxy_async();   // generic-proxy stores of A -> visible to the tensor core's operand reads
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== codebook tiles: per code tile e_hi chunks 0..DC-1, then e_lo chunks =====================
    uint32_t s = 0, ph = 1;
    bool ok = true;
    for (int t = 0; t < ntile && ok; ++t)
      for (int part = 0; part < 2 && ok; ++part)
        for (int c = 0; c < DC && ok; ++c) {
          ok = ptx::mbar_wait(b_empty(s), ph, p.dbg, 0x5601);
          if (!ok) break;
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(b_full(s), kTile);
            ptx::tma_load_2d(b_base + s * kTile, part == 0 ? &mapHi : &mapLo, b_full(s), c * 64, t * 128);
          }
          __syncwarp();
          if (++s == kNSB) { s = 0; ph ^= 1; }
        }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = idesc_f16(128, 128);
      const uint64_t ahi0 = ptx::make_smem_desc(a_hi_base, 16, 1024, ptx::kLayoutSw128);
      const uint64_t alo0 = ptx::make_smem_desc(a_lo_base, 16, 1024, ptx::kLayoutSw128);
      const uint64_t b0 = ptx::make_smem_desc(b_base, 16, 1024, ptx::kLayoutSw128);
      uint32_t s = 0, ph = 0;
      bool ok = true;
      for (int t = 0; t < ntile && ok; ++t) {
        const uint32_t b = t & 1;
        ok = ptx::mbar_wait(s_free(b), ((t >> 1) & 1) ^ 1, p.dbg, 0x5602);
        if (!ok) break;
        ptx::tc_fence_after();
        const uint32_t acc = tmem_base + b * 128;
        for (int part = 0; part < 2 && ok; ++part)
          for (int c = 0; c < DC && ok; ++c) {
            ok = ptx::mbar_wait(b_full(s), ph, p.dbg, 0x5603);
            if (!ok) break;
            ptx::tc_fence_after();
            const uint64_t db = b0 + (uint64_t)(s * (kTile >> 4));
            const uint64_t dh = ahi0 + (uint64_t)(c * (kTile >> 4)), dl = alo0 + (uint64_t)(c * (kTile >> 4));
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              ptx::tc_mma_f16(acc, dh + 2 * ks, db + 2 * ks, idesc, (part | c | ks) != 0 ? 1u : 0u);   // x_hi . e_{hi|lo}
              if (part == 0) ptx::tc_mma_f16(acc, dl + 2 * ks, db + 2 * ks, idesc, 1u);                // x_lo . e_hi
            }
            ptx::tc_commit(b_empty(s));
            if (++s == kNSB) { s = 0; ph ^= 1; }
          }
        ptx::tc_commit(s_full(b));
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== candidate scan: thread = row, one 64-column half of every score tile =====================
    const int qd = warp & 3, r = qd * 32 + lane, half = (warp - 4) >> 2;
    const int64_t row = row0 + r;
    const float inv2 = 2.0f * inv_s[r], M = marg_s[r];
    float runmin = INFINITY;
    int cnt = 0;
    bool overflow = false;
    int* ck = cand_k + (half * 128 + r) * kCap;
    float* cg = cand_g + (half * 128 + r) * kCap;
    auto push = [&](int k, float g, float thr) {
      if (overflow) return;
      if (cnt < kCap) { ck[cnt] = k; cg[cnt] = g; ++cnt; return; }
      const int n = cand_push(ck, cg, cnt, k, g, thr);
      if (n < 0) overflow = true; else cnt = n;
    };
    for (int t = 0; t < ntile; ++t) {
      const uint32_t b = t & 1;
      if (!ptx::mbar_wait(s_full(b), (t >> 1) & 1, p.dbg, 0x5604)) break;
      ptx::tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {   // 32 score columns per trip
        uint32_t ra[16], rb[16];
        const uint32_t ta = tmem_base + ((uint32_t)(qd * 32) << 16) + b * 128 + half * 64 + c * 32;
        ptx::tc_ld_32x32b_x16(ta, ra);
        ptx::tc_ld_32x32b_x16(ta + 16, rb);
        const int k0 = t * 128 + half * 64 + c * 32;
        float e2[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) *reinterpret_cast<float4*>(&e2[4 * j]) = *reinterpret_cast<const float4*>(&e2_s[k0 + 4 * j]);
        ptx::tc_wait_ld();
        float g[32];   // ||e||^2 - 2 x.e (approximate)
#pragma unroll
        for (int j = 0; j < 16; ++j) { g[j] = fmaf(-inv2, __uint_as_float(ra[j]), e2[j]); g[16 + j] = fmaf(-inv2, __uint_as_float(rb[j]), e2[16 + j]); }
        float q4[8];   // minima of the 8 groups of 4 columns
#pragma unroll
        for (int i = 0; i < 8; ++i) q4[i] = fminf(fminf(g[4 * i], g[4 * i + 1]), fminf(g[4 * i + 2], g[4 * i + 3]));
        const float m = fminf(fminf(fminf(q4[0], q4[1]), fminf(q4[2], q4[3])), fminf(fminf(q4[4], q4[5]), fminf(q4[6], q4[7])));
        // candidates of this trip against the running minimum BEFORE it (a superset of the sequential test; the final filter uses the
        // final minimum).  Taken by few lanes once the minimum has settled: the common trip is 32 FMAs + the min tree + one compare;
        // a lane with a hit looks only into the groups of 4 whose minimum passes.
        if (m <= runmin + M) {
          const float thr = fminf(runmin, m) + M;   // what is above this can never be within M of the final minimum
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (q4[i] <= thr) {
#pragma unroll
              for (int j = 4 * i; j < 4 * i + 4; ++j)
                if (g[j] <= thr) push(k0 + j, g[j], thr);
            }
        }
        runmin = fminf(runmin, m);
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(s_free(b));
    }
    half_min[half * 128 + r] = overflow ? -INFINITY : runmin;
    half_cnt[half * 128 + r] = cnt;
    scan_bar_sync();
    // ---- decide (warps of half 0): merge the two halves of the row
    if (half == 0) {
      int best_k = 0;
      if (row < p.n) {
        const float m0 = half_min[r], m1 = half_min[128 + r];
        const bool over = m0 == -INFINITY || m1 == -INFINITY;
        const float thr = fminf(m0, m1) + M;
        int nlive = 0, only = 0;
        for (int h = 0; h < 2; ++h) {
          const int n = half_cnt[h * 128 + r];
          for (int i = 0; i < n; ++i)
            if (cand_g[(h * 128 + r) * kCap + i] <= thr) { ++nlive; only = cand_k[(h * 128 + r) * kCap + i]; }
        }
        if (M < 0.f || over || nlive == 0) {
          // full exact scan: non-finite / out-of-range row (every comparison false -> code 0, like vq_kernel), candidate overflow
          const float xsq = exact_xsq<kX16>(p, row);
          float best = INFINITY;
          int bi = 0x7fffffff;
          for (int k = 0; k < p.k; ++k) {
            const float dist = exact_dist<kX16>(p, row, k, xsq);
            if (dist < best || (dist == best && k < bi)) { best = dist; bi = k; }
          }
          best_k = (unsigned)bi >= (unsigned)p.k ? 0 : bi;
          if (p.stats) atomicAdd(p.stats + 2, 1ull);
        } else if (nlive == 1) {
          best_k = only;
        } else {
          const float xsq = exact_xsq<kX16>(p, row);
          float best = INFINITY;
          int bi = 0x7fffffff;
          for (int h = 0; h < 2; ++h) {
            const int n = half_cnt[h * 128 + r];
            for (int i = 0; i < n; ++i) {
              if (!(cand_g[(h * 128 + r) * kCap + i] <= thr)) continue;
              const int k = cand_k[(h * 128 + r) * kCap + i];
              const float dist = exact_dist<kX16>(p, row, k, xsq);
              if (dist < best || (dist == best && k < bi)) { best = dist; bi = k; }   // lowest index on ties, whatever the list order
            }
          }
          best_k = (unsigned)bi >= (unsigned)p.k ? 0 : bi;
          if (p.stats) { atomicAdd(p.stats, 1ull); atomicAdd(p.stats + 1, (unsigned long long)nlive); }
        }
        p.idx[row] = (int64_t)best_k;
        if (p.hist) atomicAdd(p.hist + best_k, 1);
      }
      final_idx[r] = best_k;
    }
  } else {
    // warps 2-3: pull the rows of the CTA that follows on this SM (one wave later) into L2 while this one computes
    const int64_t nrow0 = row0 + (int64_t)p.wave_ctas * 128;
    if (nrow0 < p.n) {
      const int64_t nrows = (p.n - nrow0) < 128 ? (p.n - nrow0) : 128;
      const int64_t bytes = nrows * p.d * (kX16 ? 2 : 4);
      const char* base = reinterpret_cast<const char*>(p.x) + nrow0 * p.d * (kX16 ? 2 : 4);
      for (int64_t off = (int64_t)((warp - 2) * 32 + lane) * 128; off < bytes; off += 64 * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) { ptx::tc_fence_after(); ptx::tmem_dealloc(tmem_base, 256); }
  if (p.q) {
    // gather: a warp streams rows, 16-byte vectors, all loads of 4 rows in flight before their stores
    constexpr int kWarps = kThreads / 32;
    for (int rb = warp * 4; rb < 128; rb += kWarps * 4) {
      float4 v[4][2];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float* src = p.cb + (int64_t)final_idx[rb + u] * p.d;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int d = lane * 4 + h * 128;
          v[u][h] = (row0 + rb + u < p.n && d < p.d) ? __ldg(reinterpret_cast<const float4*>(src + d)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t gr = row0 + rb + u;
        if (gr >= p.n) break;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int d = lane * 4 + h * 128;
          if (d >= p.d) break;
          if (p.q_f32) {
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.q) + gr * p.d + d) = v[u][h];
          } else {
            act2_t* o = reinterpret_cast<act2_t*>(reinterpret_cast<act_t*>(p.q) + gr * p.d + d);
            o[0] = floats_to_act2(v[u][h].x, v[u][h].y);
            o[1] = floats_to_act2(v[u][h].z, v[u][h].w);
          }
        }
      }
    }
  }
}

// codebook -> fp16 halves scaled by 2^se (se from max |e|: max |e| 2^se in [2^13, 2^14)), + meta = {max ||e||^2, 2^-se, max |e|, out-of-range flag}
__global__ void __launch_bounds__(1024) vq_tc_prepare_kernel(const float* __restrict__ cb, const float* __restrict__ esq, int K, int D,
                                                             __half* __restrict__ ehi, __half* __restrict__ elo, float* __restrict__ meta) {
  __shared__ float red[32], red2[32];
  const int64_t total = (int64_t)K * D;
  float amax = 0.f, e2m = 0.f;
  for (int64_t i = threadIdx.x; i < total; i += blockDim.x) amax = fmaxf(amax, fabsf(cb[i]));
  for (int i = threadIdx.x; i < K; i += blockDim.x) e2m = fmaxf(e2m, esq[i]);
  amax = warp_max(amax); e2m = warp_max(e2m);
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = amax; red2[threadIdx.x >> 5] = e2m; }
  __syncthreads();
  if (threadIdx.x < 32) {
    amax = warp_max(red[threadIdx.x]); e2m = warp_max(red2[threadIdx.x]);
    if (threadIdx.x == 0) { red[0] = amax; red2[0] = e2m; }
  }
  __syncthreads();
  amax = red[0]; e2m = red2[0];
  int ex = 0;
  if (amax > 0.f) (void)frexpf(amax, &ex);
  const int se = amax > 0.f ? 14 - ex : 0;
  const float sc = ldexpf(1.0f, se);
  const bool cb_bad = !(amax >= 9.0e-13f && amax <= 1.0e12f) || !(e2m <= 3.0e38f);   // zero, huge, tiny or non-finite codebook
  if (threadIdx.x == 0) { meta[0] = e2m; meta[1] = ldexpf(1.0f, -se); meta[2] = amax; meta[3] = cb_bad ? 1.f : 0.f; }
  for (int64_t i = threadIdx.x; i < total; i += blockDim.x) {
    const float t = cb[i] * sc;
    const __half h = __float2half_rn(t);
    ehi[i] = h;
    elo[i] = __float2half_rn(t - __half2float(h));
  }
}

}  // namespace vqtc
