// K8/K9: flattened-voxel attention  O = softmax(scale * Q K^T) V (+ residual)  as ONE flash-style tcgen05 kernel.
//
// Replaces the reference's materialised (B, L, L) score tensor: tf.einsum("bhwdc,bHWDc->bhwdHWD") * scale ->
// tf.nn.softmax -> einsum with V (networks/dm3d.py:51-61; conditional_dm3d.py:171-184).  Single head, d = C.
//
//   CTA          one 128-query tile of one sample; KV tiles of BKV keys stream through a TMA ring.
//   S = Q K^T    tcgen05.mma M=128, N=BKV, K=D (A = Q tile resident in smem, B = K tile), fp32 in TMEM, two S buffers:
//                the MMAs of tile j+1 overlap the softmax of tile j.
//   softmax      4 warps, one query row per thread (TMEM lane = row): pass 1 row max, pass 2 p = exp2(s*c - m_ref) with a
//                running reference max that only moves when the new max exceeds it by > 8 (log2 units; p <= 256 stays
//                exact enough in bf16) so the O accumulator in TMEM is rescaled rarely; p -> bf16 -> smem in the
//                SWIZZLE_128B K-major layout the next MMA reads.
//   O += P V     tcgen05.mma M=128, N=D, K=BKV (A = P from smem, B = V^T tile [D][BKV], K-major), O stays in TMEM for the
//                whole key loop; epilogue O / rowsum (+ residual) -> bf16.
//   V^T          the value projection writes V transposed per sample ([B][D][L]; conv epilogue option), so both GEMMs
//                use K-major operands.
// Warps (192 threads): 0 = TMA producer, 1 = MMA issuer (+TMEM owner), 2-5 = softmax / correction / epilogue.
#include <cuda.h>
#include <math.h>
#include <new>
#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int kThreads = 192;

struct AttnParams {
  int batch, lq, lk, d;
  float scale_log2e;                 // scale * log2(e)
  const act_t* residual;     // [B][Lq][D] or null
  act_t* o;                  // [B][Lq][D]
  int* dbg;
};

__device__ __forceinline__ void tc_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void softmax_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int D, int BKV, int NST, int NPB>   // (shared-memory layout does not depend on the number of score buffers)
struct Smem {
  static constexpr int kQ = 128 * D * 2;                 // D/64 chunks of [128 rows][128 B]
  static constexpr int kK = BKV * D * 2;                 // D/64 chunks of [BKV rows][128 B]
  static constexpr int kV = D * BKV * 2;                 // BKV/64 chunks of [D rows][128 B]
  static constexpr int kP = 128 * BKV * 2;               // BKV/64 chunks of [128 rows][128 B]
  static constexpr int kBars = 1 + 4 * NST + 4 + 2 * NPB + 2;
  static_assert(NST * kK >= kQ, "the residual tile is staged in the (drained) K ring");
  static constexpr size_t kBody = kQ + (size_t)NST * (kK + kV) + (size_t)NPB * kP + kBars * 8 + 16;
  static constexpr size_t kTotal = 1024 + kBody;   // with the alignment slack (one CTA per SM)
};

// NSB = score buffers in TMEM (2: Q K^T of tile j + 1 overlaps the whole softmax of tile j; 1: it overlaps everything after
// the softmax warps' load of the row, which is enough when MINB = 2 CTAs share the SM and interleave their phases)
template <int D, int BKV, int NST, int NPB, int NSB, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
flash_attn_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                  const __grid_constant__ CUtensorMap mapVt, const __grid_constant__ CUtensorMap mapO,
                  const __grid_constant__ CUtensorMap mapR, const AttnParams p) {
  using SM = Smem<D, BKV, NST, NPB>;
  static_assert(D % 64 == 0 && D <= 256 && BKV % 64 == 0 && BKV <= 128, "tile shape");
  constexpr int kDC = D / 64, kKC = BKV / 64;
  constexpr uint32_t kOCol = NSB * BKV;                             // TMEM: S0 | (S1 |) O
  constexpr uint32_t kTmemCols = (NSB * BKV + D) <= 128 ? 128 : ((NSB * BKV + D) <= 256 ? 256 : 512);
  static_assert(kTmemCols * MINB <= 512, "co-resident CTAs share the SM's 512 TMEM columns");
  // two CTAs per SM leave no room for 1 KB of alignment slack (2 x (kBody + 1 KB reserved) = 228 KB - 1.7 KB): that variant is
  // launched with kBody bytes and relies on the 1024-byte alignment of the dynamic window (no static shared memory), checked here
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  if (MINB > 1 && smem != smem_raw) {
    if (threadIdx.x == 0 && p.dbg) atomicExch(p.dbg, 0x5701);
    return;
  }
  const uint32_t q_base = ptx::smem_u32(smem);
  const uint32_t k_base = q_base + SM::kQ;
  const uint32_t v_base = k_base + NST * SM::kK;
  const uint32_t p_base = v_base + NST * SM::kV;
  uint8_t* p_ptr = smem + SM::kQ + NST * (SM::kK + SM::kV);
  uint64_t* bars = reinterpret_cast<uint64_t*>(p_ptr + NPB * SM::kP);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + SM::kBars);
  const uint32_t bar_base = ptx::smem_u32(bars);
  const uint32_t q_full = bar_base;
  auto k_full = [&](int s) { return bar_base + 8u * (1 + s); };
  auto k_empty = [&](int s) { return bar_base + 8u * (1 + NST + s); };
  auto v_full = [&](int s) { return bar_base + 8u * (1 + 2 * NST + s); };
  auto v_empty = [&](int s) { return bar_base + 8u * (1 + 3 * NST + s); };
  auto s_full = [&](int b) { return bar_base + 8u * (1 + 4 * NST + b); };
  auto s_free = [&](int b) { return bar_base + 8u * (1 + 4 * NST + 2 + b); };
  auto p_full = [&](int b) { return bar_base + 8u * (1 + 4 * NST + 4 + b); };
  auto p_free = [&](int b) { return bar_base + 8u * (1 + 4 * NST + 4 + NPB + b); };
  const uint32_t o_done = bar_base + 8u * (1 + 4 * NST + 4 + 2 * NPB);
  const uint32_t res_full = bar_base + 8u * (1 + 4 * NST + 4 + 2 * NPB + 1);

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 128, n = blockIdx.y;
  const int ntile = (p.lk + BKV - 1) / BKV;

  if (threadIdx.x == 0) {
    ptx::mbar_init(q_full, 1);
    for (int s = 0; s < NST; ++s) {
      ptx::mbar_init(k_full(s), 1); ptx::mbar_init(k_empty(s), 1); ptx::mbar_init(v_full(s), 1); ptx::mbar_init(v_empty(s), 1);
    }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(s_full(b), 1); ptx::mbar_init(s_free(b), 4); }
    for (int b = 0; b < NPB; ++b) { ptx::mbar_init(p_full(b), 4); ptx::mbar_init(p_free(b), 1); }
    ptx::mbar_init(o_done, 1);
    ptx::mbar_init(res_full, 1);
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&mapO);
    ptx::prefetch_tmap(&mapQ); ptx::prefetch_tmap(&mapK); ptx::prefetch_tmap(&mapVt);
  }
  if (warp == 1) {
    ptx::tmem_alloc(ptx::smem_u32(tmem_ptr_smem), kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      ptx::mbar_expect_tx(q_full, SM::kQ);
      for (int c = 0; c < kDC; ++c) ptx::tma_load_3d(q_base + c * (128 * 128), &mapQ, q_full, c * 64, q0, n);
    }
    __syncwarp();
    uint32_t s = 0, ph = 1;
    for (int j = 0; j < ntile; ++j) {
      if (!ptx::mbar_wait(k_empty(s), ph, p.dbg, 21)) break;
      if (ptx::elect_one()) {
        ptx::mbar_expect_tx(k_full(s), SM::kK);
        for (int c = 0; c < kDC; ++c) ptx::tma_load_3d(k_base + s * SM::kK + c * (BKV * 128), &mapK, k_full(s), c * 64, j * BKV, n);
      }
      __syncwarp();
      if (!ptx::mbar_wait(v_empty(s), ph, p.dbg, 22)) break;
      if (ptx::elect_one()) {
        ptx::mbar_expect_tx(v_full(s), SM::kV);
        for (int c = 0; c < kKC; ++c) ptx::tma_load_3d(v_base + s * SM::kV + c * (D * 128), &mapVt, v_full(s), j * BKV + c * 64, 0, n);
      }
      __syncwarp();
      if (++s == NST) { s = 0; ph ^= 1; }
    }
    if (p.residual) {
      // residual tile -> the K ring once every Q K^T has drained it (same [chunk][128 rows][128 B] layout as the Q tile);
      // it lands while the last softmax / P V are still running
      bool okr = true;
      for (int i = 0; i < NST && okr; ++i) {
        okr = ptx::mbar_wait(k_empty(s), ph, p.dbg, 32);
        if (++s == NST) { s = 0; ph ^= 1; }
      }
      if (okr && ptx::elect_one()) {
        ptx::mbar_expect_tx(res_full, SM::kQ);
        for (int c = 0; c < kDC; ++c) ptx::tma_load_3d(k_base + c * (128 * 128), &mapR, res_full, c * 64, q0, n);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc_s = ptx::make_idesc_act(128, BKV);
    constexpr uint32_t idesc_o = ptx::make_idesc_act(128, D);
    const uint64_t dq = ptx::make_smem_desc(q_base, 16, 1024, ptx::kLayoutSw128);
    const uint64_t dk = ptx::make_smem_desc(k_base, 16, 1024, ptx::kLayoutSw128);
    const uint64_t dv = ptx::make_smem_desc(v_base, 16, 1024, ptx::kLayoutSw128);
    const uint64_t dp = ptx::make_smem_desc(p_base, 16, 1024, ptx::kLayoutSw128);
    bool ok = ptx::mbar_wait(q_full, 0, p.dbg, 23);
    auto issue_qk = [&](int j) {   // S[j&1] = Q K_j^T
      const int s = j % NST;
      ok = ok && ptx::mbar_wait(k_full(s), (j / NST) & 1, p.dbg, 24);
      if (j >= NSB) ok = ok && ptx::mbar_wait(s_free(j % NSB), ((j / NSB) - 1) & 1, p.dbg, 25);
      if (!ok) return;
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint32_t acc = tmem_base + (uint32_t)(j % NSB) * BKV;
#pragma unroll
        for (int c = 0; c < kDC; ++c) {
          const uint64_t a = dq + (uint64_t)(c * ((128 * 128) >> 4));
          const uint64_t b = dk + (uint64_t)((s * SM::kK + c * (BKV * 128)) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) ptx::tc_mma_f16(acc, a + 2 * k, b + 2 * k, idesc_s, (c | k) != 0 ? 1u : 0u);
        }
        ptx::tc_commit(k_empty(s));
        ptx::tc_commit(s_full(j % NSB));
      }
      __syncwarp();
    };
    issue_qk(0);
    for (int j = 0; j < ntile && ok; ++j) {
      if (j + 1 < ntile) issue_qk(j + 1);
      const int s = j % NST, pb = j % NPB;
      ok = ok && ptx::mbar_wait(p_full(pb), (j / NPB) & 1, p.dbg, 26);
      ok = ok && ptx::mbar_wait(v_full(s), (j / NST) & 1, p.dbg, 27);
      if (!ok) break;
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint32_t acc = tmem_base + kOCol;
#pragma unroll
        for (int c = 0; c < kKC; ++c) {
          const uint64_t a = dp + (uint64_t)((pb * SM::kP + c * (128 * 128)) >> 4);
          const uint64_t b = dv + (uint64_t)((s * SM::kV + c * (D * 128)) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) ptx::tc_mma_f16(acc, a + 2 * k, b + 2 * k, idesc_o, (j | c | k) != 0 ? 1u : 0u);
        }
        ptx::tc_commit(v_empty(s));
        ptx::tc_commit(p_free(pb));
        ptx::tc_commit(o_done);
      }
      __syncwarp();
    }
  } else {
    // ===================== softmax / correction / epilogue (TMEM lane quarter = warp % 4) =====================
    const int qd = warp & 3;
    const int r = qd * 32 + lane;                       // query row within the tile
    const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
    float m_ref = -INFINITY, l = 0.f;                   // reference max (log2 units) and running sum
    bool ok = true;
    for (int j = 0; j < ntile && ok; ++j) {
      const int sb = j % NSB, pb = j % NPB;
      ok = ptx::mbar_wait(s_full(sb), (j / NSB) & 1, p.dbg, 28);
      if (!ok) break;
      ptx::tc_fence_after();
      const uint32_t s_addr = lane_addr + (uint32_t)sb * BKV;
      const int kvalid = p.lk - j * BKV;                // keys of this tile that exist
      // ---- the whole score row of this tile -> registers in one round trip (BKV loads in flight, one wait): the TMEM buffer is
      // free for Q K^T (j + 2) before the exponentials start, and the row is read once instead of twice
      uint32_t sv[BKV];
#pragma unroll
      for (int c0 = 0; c0 < BKV; c0 += 16) ptx::tc_ld_32x32b_x16(s_addr + c0, *reinterpret_cast<uint32_t(*)[16]>(&sv[c0]));
      ptx::tc_wait_ld();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(s_free(sb));
      if (kvalid < BKV) {   // last tile only (warp-uniform): keys past Lk score -inf, exp2 makes them 0
#pragma unroll
        for (int i = 0; i < BKV; ++i)
          if (i >= kvalid) sv[i] = 0xff800000u;
      }
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int i = 0; i < BKV; i += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) mx4[u] = fmaxf(mx4[u], __uint_as_float(sv[i + u]));
      }
      float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])) * p.scale_log2e;
      // ---- reference max update + (rare) rescale of the O accumulator
      float factor = 1.f;
      const bool grow = mx > m_ref + 8.f;               // first tile: m_ref = -inf
      if (grow) {
        factor = (m_ref == -INFINITY) ? 0.f : ex2(m_ref - mx);
        m_ref = mx;
        l *= factor;
      }
      if (j > 0 && __any_sync(0xffffffffu, grow)) {
        ok = ptx::mbar_wait(o_done, (j - 1) & 1, p.dbg, 29);   // PV(j-1) has landed in TMEM
        if (!ok) break;
        ptx::tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < D; c0 += 16) {
          uint32_t rr[16];
          ptx::tc_ld_32x32b_x16(lane_addr + kOCol + c0, rr);
          ptx::tc_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; ++i) rr[i] = __float_as_uint(__uint_as_float(rr[i]) * factor);
          tc_st_32x32b_x16(lane_addr + kOCol + c0, rr);
        }
        tc_wait_st();
        ptx::tc_fence_before();
      }
      // ---- p = exp2(s*c - m_ref) -> 16-bit (in place: two per register)
      float ls4[4] = {0.f, 0.f, 0.f, 0.f};
      const float nm = -m_ref;
#pragma unroll
      for (int i = 0; i < BKV; i += 2) {
        const float p0 = ex2(fmaf(__uint_as_float(sv[i]), p.scale_log2e, nm));
        const float p1 = ex2(fmaf(__uint_as_float(sv[i + 1]), p.scale_log2e, nm));
#ifdef B200DM_ACT_FP16
        // l sums the ROUNDED p, the weights P.V consumes, so that they are normalised exactly: in fp16, p < 2^-25 rounds to
        // 0, and summing the unrounded p would shrink the output by (sum of the flushed p) / l -- 2.8e-3 for 131072 keys 25.5
        // binades below the row maximum.  (Shifting p up instead does not help: the tensor cores' fp32 accumulation of P.V
        // drops products that far below the running O.)  bf16 has fp32's exponent range; its p do not underflow.
        const act2_t h = floats_to_act2(p0, p1);
        const float2 hf = act2_to_float2(h);
        ls4[(i >> 1) & 3] += hf.x + hf.y;
#else
        ls4[(i >> 1) & 3] += p0 + p1;
        const act2_t h = floats_to_act2(p0, p1);
#endif
        memcpy(&sv[i >> 1], &h, 4);
      }
      l += (ls4[0] + ls4[1]) + (ls4[2] + ls4[3]);
      // ---- the P buffer must have been consumed by PV(j - NPB)
      if (j >= NPB) {
        ok = ptx::mbar_wait(p_free(pb), ((j / NPB) - 1) & 1, p.dbg, 30);
        if (!ok) break;
      }
      // ---- -> smem (SWIZZLE_128B, K-major: chunk of 64 keys = [128 rows][128 B])
      uint8_t* prow = p_ptr + pb * SM::kP + r * 128;
#pragma unroll
      for (int u = 0; u < BKV / 8; ++u) {               // 16-byte units of 8 keys
        uint8_t* chunk = prow + (u >> 3) * (128 * 128);
        *reinterpret_cast<uint4*>(chunk + (((u & 7) ^ (r & 7)) << 4)) = make_uint4(sv[4 * u], sv[4 * u + 1], sv[4 * u + 2], sv[4 * u + 3]);
      }
      ptx::fence_proxy_async();                         // generic-proxy smem writes -> visible to the tensor-core (async) proxy
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(p_full(pb));
    }
    // ---- epilogue: O / l (+ residual) -> bf16
    if (ok) ok = ptx::mbar_wait(o_done, (ntile - 1) & 1, p.dbg, 31);
    ptx::tc_fence_after();
    // O tile -> bf16 in the (idle) Q tile's smem, SWIZZLE_128B -> one TMA store per 64-column chunk: whole 128-byte rows,
    // rows past Lq clipped by the TMA unit (row-per-thread global stores touch 32 lines per instruction)
    if (ok && p.residual) ok = ptx::mbar_wait(res_full, 0, p.dbg, 33);
    if (ok) {
      const float inv = 1.f / l;
      uint8_t* q_ptr = smem;
      const uint8_t* r_ptr = smem + SM::kQ;
#pragma unroll 1
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t ra[16], rb[16];
        ptx::tc_ld_32x32b_x16(lane_addr + kOCol + c0, ra);
        ptx::tc_ld_32x32b_x16(lane_addr + kOCol + c0 + 16, rb);
        ptx::tc_wait_ld();
        float v[32];
#pragma unroll
        for (int i = 0; i < 16; ++i) { v[i] = __uint_as_float(ra[i]) * inv; v[16 + i] = __uint_as_float(rb[i]) * inv; }
        const uint32_t base = (uint32_t)(c0 >> 6) * (128 * 128) + (uint32_t)r * 128u;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t o = base + (uint32_t)(((((c0 & 63) >> 3) + u) ^ (r & 7)) << 4);
          if (p.residual) {
            float a[8];
            unpack8(*reinterpret_cast<const bf16x8*>(r_ptr + o), a);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[8 * u + i] += a[i];
          }
          *reinterpret_cast<bf16x8*>(q_ptr + o) = pack8(*reinterpret_cast<float(*)[8]>(&v[8 * u]));
        }
      }
      ptx::fence_proxy_async();
      softmax_bar_sync();
      if (threadIdx.x == 64) {
        for (int c = 0; c < kDC; ++c)
          asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::
                           "l"(reinterpret_cast<uint64_t>(&mapO)), "r"(q_base + c * (128 * 128)), "r"(c * 64), "r"(q0), "r"(n)
                       : "memory");
        ptx::bulk_commit_group();
        ptx::bulk_wait_read_all();
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ld = row stride in elements (0 = d0: contiguous rows); lets Q / K be column blocks of one wider projection output
int encode3(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t b0, uint32_t b1, uint64_t ld = 0) {
  EncodeTiledFn enc = b2_encode_tiled_fn();
  if (!enc) { b200dm_set_error("attention: cuTensorMapEncodeTiled unavailable"); return B200DM_ERR_CUDA; }
  if (ld == 0) ld = d0;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {ld * 2, ld * d1 * 2};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(m, kTmapAct16, 3, const_cast<void*>(ptr), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { b200dm_set_error("attention: cuTensorMapEncodeTiled failed: %d (dims %llu,%llu,%llu box %u,%u)", (int)r,
                                            (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, b0, b1); return B200DM_ERR_CUDA; }
  return B200DM_OK;
}

}  // namespace

struct b200dm_attn_plan {
  b200dm_attn_desc desc;
  AttnParams p;
  CUtensorMap mapQ, mapK, mapVt, mapO, mapR;
  int bkv;
  size_t smem;
  double flops;
};

int* b200dm_dbg_flag_ptr();

template <int D, int BKV, int NST, int NPB, int NSB, int MINB>
static int launch_attn(const b200dm_attn_plan* pl, cudaStream_t s) {
  auto kern = flash_attn_kernel<D, BKV, NST, NPB, NSB, MINB>;
  constexpr size_t kSmem = MINB > 1 ? Smem<D, BKV, NST, NPB>::kBody : Smem<D, BKV, NST, NPB>::kTotal;
  static_assert(MINB * (kSmem + 1024) <= 233472, "co-resident CTAs fit the SM's shared memory");
  static bool attr_set = false;
  if (!attr_set) {
    B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
    if (MINB > 1) B2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    attr_set = true;
  }
  dim3 grid((pl->desc.lq + 127) / 128, pl->desc.batch);
  B2_CHECK_CUDA(b2_launch(kern, grid, dim3(kThreads), kSmem, s, pl->mapQ, pl->mapK, pl->mapVt, pl->mapO, pl->mapR, pl->p));
  return B200DM_OK;
}

extern "C" int b200dm_attention_plan_create(const b200dm_attn_desc* d, const void* q, const void* k, const void* vt,
                                            const void* residual, void* o, b200dm_attn_plan** out) {
  B2_CHECK_ARG(out, "attention_plan_create: null out");
  *out = nullptr;
  B2_CHECK_ARG(d && q && k && vt && o, "attention_plan_create: null argument");
  B2_CHECK_ARG(d->batch > 0 && d->lq > 0 && d->lk > 0, "attention_plan_create: empty problem");
  B2_CHECK_ARG(d->d == 64 || d->d == 128 || d->d == 256, "attention_plan_create: head dim %d unsupported (64, 128, 256)", d->d);
  B2_CHECK_ARG(d->lk % 8 == 0, "attention_plan_create: Lk must be a multiple of 8 (16-byte rows of V^T)");
  b200dm_attn_plan* pl = new (std::nothrow) b200dm_attn_plan();
  B2_CHECK_ARG(pl, "attention_plan_create: out of memory");
  pl->desc = *d;
  pl->bkv = d->d == 256 ? 64 : 128;
  // reserved[0] / reserved[1]: row strides (elements) of q / k when they are column blocks of a wider tensor (0 = D)
  B2_CHECK_ARG(d->reserved[0] >= 0 && d->reserved[1] >= 0 && d->reserved[0] % 8 == 0 && d->reserved[1] % 8 == 0 &&
                   (d->reserved[0] == 0 || d->reserved[0] >= d->d) && (d->reserved[1] == 0 || d->reserved[1] >= d->d),
               "attention_plan_create: q / k row strides must be 0 or multiples of 8 >= D");
  int rc = encode3(&pl->mapQ, q, d->d, d->lq, d->batch, 64, 128, (uint64_t)d->reserved[0]);
  if (!rc) rc = encode3(&pl->mapK, k, d->d, d->lk, d->batch, 64, pl->bkv, (uint64_t)d->reserved[1]);
  if (!rc) rc = encode3(&pl->mapVt, vt, d->lk, d->d, d->batch, 64, d->d);
  if (!rc) rc = encode3(&pl->mapO, o, d->d, d->lq, d->batch, 64, 128);
  if (!rc) rc = encode3(&pl->mapR, residual ? residual : o, d->d, d->lq, d->batch, 64, 128);
  if (rc) { delete pl; return rc; }
  pl->p.batch = d->batch; pl->p.lq = d->lq; pl->p.lk = d->lk; pl->p.d = d->d;
  pl->p.scale_log2e = d->scale * 1.4426950408889634f;
  pl->p.residual = (const act_t*)residual;
  pl->p.o = (act_t*)o;
  pl->p.dbg = b200dm_dbg_flag_ptr();
  pl->flops = 4.0 * d->batch * (double)d->lq * d->lk * d->d;
  *out = pl;
  return B200DM_OK;
}

extern "C" int b200dm_attention_plan_run(b200dm_attn_plan* pl, void* stream) {
  B2_CHECK_ARG(pl, "attention_plan_run: null plan");
  cudaStream_t s = (cudaStream_t)stream;
  switch (pl->desc.d) {
    // d = 64 (cfg-4, L = 32768): the exponentials (MUFU, 1024 cycles per 128 x 128 tile) outweigh the MMAs (640), and one CTA's
    // softmax -> P V -> next softmax chain leaves both pipes idle half of the time: two CTAs per SM (112 KB, 256 TMEM columns each)
    case 64: return launch_attn<64, 128, 2, 1, 1, 2>(pl, s);
    case 128: return launch_attn<128, 128, 2, 1, 2, 1>(pl, s);
    case 256: return launch_attn<256, 64, 2, 1, 2, 1>(pl, s);
  }
  b200dm_set_error("attention_plan_run: unsupported head dim");
  return B200DM_ERR_UNSUPPORTED;
}

extern "C" void b200dm_attention_plan_destroy(b200dm_attn_plan* p) { delete p; }
extern "C" double b200dm_attention_plan_flops(const b200dm_attn_plan* p) { return p ? p->flops : 0.0; }
