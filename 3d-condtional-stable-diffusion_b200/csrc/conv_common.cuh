// Shared between the two implicit-GEMM conv kernels: launch parameters and the fused epilogue.
#pragma once
#include "common.cuh"
#include "ptx.cuh"
#include "update_math.cuh"

struct ConvParams {
  int mode, batch;
  int in_d, in_h, in_w;
  int out_d, out_h, out_w;
  int m_d, m_h, m_w;                 // M-space extent (== out for DIRECT / GEMM, == in for PARITY)
  int box_w, box_h, box_d, box_n;    // product == 128
  int tiles_w, tiles_h, tiles_d, tiles_n;
  int nch0, nch1, ntaps, ksize, stride, pad;
  int ksteps0_last, ksteps1_last;    // K=16 MMA steps that hold real channels in the LAST 64-channel chunk of each segment (1..4)
  // halo kernel: a 1^3 conv of two more segments (the ResidualBlock shortcut of [x | skip]) accumulated after the 3^3 chunks,
  // centre tap only (b200dm_conv_plan_set_shortcut); sc_nch0 = 0: none
  int sc_nch0, sc_nch1, sc_ksteps0_last, sc_ksteps1_last;
  int c_out, n_pad;
  int act, post_act, y_f32, transposed_store;
  int chan_bias_rows;
  int halo_td, halo_tiles_per_ntile, halo_ntn, halo_total_tiles;   // halo kernel only
  int tma_epi;                       // staged epilogue: bf16 tile -> swizzled smem -> TMA store (residual tile TMA-loaded)
  int swap_ab;                       // transposed store by operand swap: D^T = W X^T (TMEM lane = channel, column = voxel)
  int ksplit;                        // igemm split-K: cluster of ksplit CTAs per tile, each owns a K range (0/1 = off)
  const float* bias;
  const float* out_scale;            // optional per-channel affine applied after the bias adds (a folded BatchNorm of the
  const float* out_shift;            // CONSUMER: y = act(scale * (acc + bias + temb) + shift)), fp32[c_out]
  const float* chan_bias;
  const int* t_dev;
  const act_t* residual;
  const act_t* prelu_alpha;  // (d,h,w,c) bf16, no batch dim
  void* y;
  int* dbg;
  long long* trace;                  // optional per-role clock64 timeline of CTA 0 (tuning aid), else nullptr
  // fused reverse-diffusion update (the U-Net's output conv on the sampling graph, b200dm_conv_plan_set_fused_update): the
  // epilogue turns its eps tile into x_{t-1} = step(x_t, eps, Philox noise) and stores that (fp32 through the y map + a
  // 16-bit copy for the next step's input conv) instead of eps -- the fp32 eps round trip through HBM and the update
  // kernel's launch disappear.  upd_x = x_t (fp32, the output's geometry); nullptr = off.
  const float* upd_x;
  b200dm_update_desc upd;
};

// Output-side tensor maps of the staged (TMA-store) epilogue: y[parity] (parity 0 only outside PARITY mode), r = residual.
struct ConvOutMaps {
  CUtensorMap y[8];
  CUtensorMap r;
};

// timeline regions (each kTraceRegion entries): 0 = MMA issuer, 1 = epilogue warp 4, 2 = slab producer, 3 = weight producer
constexpr int kTraceRegion = 2048;
__device__ __forceinline__ void trace_ev(const ConvParams& p, int region, int& idx, int tag) {
  if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && idx < kTraceRegion - 1) {
    p.trace[region * kTraceRegion + idx] = (clock64() << 8) | (long long)(tag & 0xff);
    ++idx;
  }
}

__device__ __forceinline__ float bf(const act_t v) { return act_to_float(v); }

// The epilogue's per-column terms on 16 values: + cb[col0 + j] (a global chan_bias row, only when a tile spans several
// samples) -> * sc[j] -> + bs[j] (sc / bs: staged in shared memory once per tile, see conv_epilogue16).  nullptr = term absent.
__device__ __forceinline__ void bias_scale16(float (&v)[16], const float* cb, int col0, const float* sc, const float* bs) {
  if (cb) {
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
      const float4 b4 = __ldg(reinterpret_cast<const float4*>(cb + col0 + j));
      v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
    }
  }
  if (sc) {
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
      const float4 s4 = *reinterpret_cast<const float4*>(sc + j);
      v[j] *= s4.x; v[j + 1] *= s4.y; v[j + 2] *= s4.z; v[j + 3] *= s4.w;
    }
  }
  if (bs) {
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
      const float4 b4 = *reinterpret_cast<const float4*>(bs + j);
      v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
    }
  }
}


// Byte offset of 16-byte unit `u` of row `r` in a tile of `row_bytes`-byte rows (128, 64 or 32) as a tensor map with
// CU_TENSOR_MAP_SWIZZLE_128B / 64B / 32B lays it out in shared memory: the unit index is XORed with bits 7.. of the row's address.
__device__ __forceinline__ uint32_t swizzle_off(uint32_t row_bytes, int r, int u) {
  const int sw = row_bytes == 128 ? r & 7 : (row_bytes == 64 ? (r >> 1) & 3 : (r >> 2) & 1);
  return (uint32_t)r * row_bytes + (uint32_t)((u ^ sw) << 4);
}

// Epilogue for 16 consecutive accumulator columns of one output voxel (thread = TMEM lane = GEMM row):
//   + bias[co] + chan_bias[t][n][co]  ->  * out_scale[co] + out_shift[co]  ->  PReLU(alpha[voxel][co])  ->  act  ->
//   + residual  ->  post_act  ->  store
// `bs`: 16 floats in SHARED memory = bias (+ chan_bias when it is uniform over the tile) for these columns, staged once
// per tile (a per-chunk __ldg round trip made the epilogue as long as the tile's MMA phase); with an output affine
// `sc` holds the 16 scales and `bs` holds scale * bias + shift.  `cb`: per-row global chan_bias pointer, only when a
// tile spans several samples.
__device__ __forceinline__ void conv_epilogue16(const ConvParams& p, const uint32_t (&rr)[16], int col0, int n, int64_t vox,
                                                int64_t vox_per, int64_t row_off, const float* bs, const float* cb,
                                                const float* sc = nullptr, const bf16x8* rpre = nullptr) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]);
  const int ncol = (p.c_out - col0) < 16 ? (p.c_out - col0) : 16;
  if (ncol == 16 && !p.transposed_store) {
    // vector path: 16 channels = 32 B bf16 / 64 B fp32 per thread
    bias_scale16(v, cb, col0, sc, bs);
    if (p.prelu_alpha) {
      float a[16];
      const act_t* ap = p.prelu_alpha + vox * p.c_out + col0;
      unpack8(*reinterpret_cast<const bf16x8*>(ap), *reinterpret_cast<float(*)[8]>(&a[0]));
      unpack8(*reinterpret_cast<const bf16x8*>(ap + 8), *reinterpret_cast<float(*)[8]>(&a[8]));
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f) + a[j] * fminf(v[j], 0.f);
    }
    if (p.act != B200DM_ACT_NONE) {
      apply_act_vec(v, p.act);
    }
    if (p.residual) {
      float a[16];
      if (rpre) {   // residual already in registers (prefetched while the MMAs ran)
        unpack8(rpre[0], *reinterpret_cast<float(*)[8]>(&a[0]));
        unpack8(rpre[1], *reinterpret_cast<float(*)[8]>(&a[8]));
      } else {
        const act_t* rp = p.residual + row_off + col0;
        unpack8(*reinterpret_cast<const bf16x8*>(rp), *reinterpret_cast<float(*)[8]>(&a[0]));
        unpack8(*reinterpret_cast<const bf16x8*>(rp + 8), *reinterpret_cast<float(*)[8]>(&a[8]));
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] += a[j];
    }
    if (p.post_act != B200DM_ACT_NONE) {
      apply_act_vec(v, p.post_act);
    }
    if (p.y_f32) {
      float* yo = reinterpret_cast<float*>(p.y) + row_off + col0;
#pragma unroll
      for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(yo + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
      act_t* yo = reinterpret_cast<act_t*>(p.y) + row_off + col0;
      *reinterpret_cast<bf16x8*>(yo) = pack8(*reinterpret_cast<float(*)[8]>(&v[0]));
      *reinterpret_cast<bf16x8*>(yo + 8) = pack8(*reinterpret_cast<float(*)[8]>(&v[8]));
    }
  } else {
    // scalar path: ragged channel tail (e.g. C_out = 1) or per-sample transposed store
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (j < ncol) {
        const int col = col0 + j;
        float x = v[j];
        if (cb) x += __ldg(cb + col);
        if (sc) x *= sc[j];
        if (bs) x += bs[j];
        if (p.prelu_alpha) { const float a = bf(p.prelu_alpha[vox * p.c_out + col]); x = fmaxf(x, 0.f) + a * fminf(x, 0.f); }
        x = apply_act(x, p.act);
        if (p.residual) x += bf(p.residual[row_off + col]);
        x = apply_act(x, p.post_act);
        const int64_t o = p.transposed_store ? ((int64_t)n * p.c_out + col) * vox_per + vox : row_off + col;
        if (p.y_f32) reinterpret_cast<float*>(p.y)[o] = x;
        else reinterpret_cast<act_t*>(p.y)[o] = float_to_act(x);
      }
    }
  }
}

// Staged epilogue for 16 consecutive columns of GEMM row `r` (c_local = first column within the 64-column group):
// same arithmetic as the vector path of conv_epilogue16 (no PReLU / fp32 / transposed forms -- the host never selects
// the staged path for those), residual read from the TMA-loaded swizzled tile `rs`, result written as bf16 into the
// swizzled staging tile `stg` ([128 rows][128 B], 16-byte chunk index XOR (row & 7) = CU_TENSOR_MAP_SWIZZLE_128B).
__device__ __forceinline__ void conv_epilogue16_staged(const ConvParams& p, const uint32_t (&rr)[16], int r, int c_local, int col0,
                                                       const float* bs, const float* cb, const float* sc, const uint8_t* rs,
                                                       uint8_t* stg, bool has_rpre = false, const bf16x8* rpre = nullptr,
                                                       bool row64 = false) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]);
  bias_scale16(v, cb, col0, sc, bs);
  if (p.act != B200DM_ACT_NONE) {
    apply_act_vec(v, p.act);
  }
  // 128-byte rows (64 channels, SWIZZLE_128B: chunk ^ (row & 7)) or 64-byte rows (32 channels, SWIZZLE_64B: chunk ^ ((row >> 1) & 3))
  const int ch = c_local >> 3;
  const uint32_t row_bytes = row64 ? 64u : 128u;
  const uint32_t o0 = swizzle_off(row_bytes, r, ch), o1 = swizzle_off(row_bytes, r, ch + 1);
  if (rs) {
    float a[16];
    unpack8(*reinterpret_cast<const bf16x8*>(rs + o0), *reinterpret_cast<float(*)[8]>(&a[0]));
    unpack8(*reinterpret_cast<const bf16x8*>(rs + o1), *reinterpret_cast<float(*)[8]>(&a[8]));
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] += a[j];
  } else if (has_rpre) {   // residual row already in registers (rpre is dereferenced only here: stays in registers)
    float a[16];
    unpack8(rpre[0], *reinterpret_cast<float(*)[8]>(&a[0]));
    unpack8(rpre[1], *reinterpret_cast<float(*)[8]>(&a[8]));
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] += a[j];
  }
  if (p.post_act != B200DM_ACT_NONE) {
    apply_act_vec(v, p.post_act);
  }
  *reinterpret_cast<bf16x8*>(stg + o0) = pack8(*reinterpret_cast<float(*)[8]>(&v[0]));
  *reinterpret_cast<bf16x8*>(stg + o1) = pack8(*reinterpret_cast<float(*)[8]>(&v[8]));
}

// fp32 form of the staged epilogue: 16 columns = 64 bytes = four 16-byte units of a [128 rows][128 B] tile that holds
// 32 fp32 columns (c_local = 0 or 16 within the 32-column group); bias / scale / act / register residual as above.
__device__ __forceinline__ void conv_epilogue16_staged_f32(const ConvParams& p, const uint32_t (&rr)[16], int r, int c_local,
                                                           const float* bs, const float* sc, uint8_t* stg, bool has_rpre,
                                                           const bf16x8* rpre) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]);
  bias_scale16(v, nullptr, 0, sc, bs);
  if (p.act != B200DM_ACT_NONE) {
    apply_act_vec(v, p.act);
  }
  if (has_rpre) {
    float a[16];
    unpack8(rpre[0], *reinterpret_cast<float(*)[8]>(&a[0]));
    unpack8(rpre[1], *reinterpret_cast<float(*)[8]>(&a[8]));
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] += a[j];
  }
  if (p.post_act != B200DM_ACT_NONE) {
    apply_act_vec(v, p.post_act);
  }
#pragma unroll
  for (int u = 0; u < 4; ++u)
    *reinterpret_cast<float4*>(stg + swizzle_off(128, r, (c_local >> 2) + u)) = make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
}

// Fused-update form of the fp32 staged epilogue: the 16 accumulator columns of this thread's row are eps_hat.  x_t of the same
// 128 rows x 16 columns has been TMA-loaded INTO the fp32 staging tile (64-byte rows, SWIZZLE_64B; completion on mbarrier
// `xbar`): each thread reads its 16 values from the very chunks it then overwrites with x_{t-1}; a second tile of 32-byte rows
// (SWIZZLE_32B) takes the copy rounded to the 16-bit storage type.  The noise comes from the Philox stream of the stand-alone
// update kernel (counter = element / 4 of the sample, step = t, sample = global sample index) and is generated BEFORE the
// wait on the x_t tile, so the load's latency hides behind it.
__device__ __forceinline__ bool upd_epilogue16(const ConvParams& p, const uint32_t (&rr)[16], int r, const float* bs, const float* sc,
                                               const upd::Coef& k, bool gen, uint32_t ctr0, uint32_t sample, uint64_t seed,
                                               uint8_t* stg, uint8_t* stg16, uint32_t xbar, uint32_t xphase) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]);
  bias_scale16(v, nullptr, 0, sc, bs);
  float z[16];
  if (gen) {
#pragma unroll
    for (int q = 0; q < 4; ++q) upd::normal4(ctr0 + q, (uint32_t)k.t, sample, 0u, seed, *reinterpret_cast<float(*)[4]>(&z[4 * q]));
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) z[j] = 0.0f;
  }
  if (!ptx::mbar_wait(xbar, xphase, p.dbg, 17)) return false;
  float x[16], y[16];
#pragma unroll
  for (int u = 0; u < 4; ++u) *reinterpret_cast<float4*>(&x[4 * u]) = *reinterpret_cast<const float4*>(stg + swizzle_off(64, r, u));
  upd::step_vec(k, p.upd.sampler, x, v, z, y);
#pragma unroll
  for (int u = 0; u < 4; ++u) *reinterpret_cast<float4*>(stg + swizzle_off(64, r, u)) = make_float4(y[4 * u], y[4 * u + 1], y[4 * u + 2], y[4 * u + 3]);
  *reinterpret_cast<bf16x8*>(stg16 + swizzle_off(32, r, 0)) = pack8(*reinterpret_cast<float(*)[8]>(&y[0]));
  *reinterpret_cast<bf16x8*>(stg16 + swizzle_off(32, r, 1)) = pack8(*reinterpret_cast<float(*)[8]>(&y[8]));
  return true;
}

// Stage bias[col] (+ chan_bias row `cbrow` when given) for columns [col_base, col_base + ncols) into shared memory.
// With an output affine, dst_scale[c] = scale and dst[c] = scale * bias + shift.
// Called by the epilogue threads (tid 0..nthreads-1); columns past c_out read as 0.
__device__ __forceinline__ void stage_bias(const ConvParams& p, float* dst, float* dst_scale, int col_base, int ncols,
                                           const float* cbrow, int tid, int nthreads = 128) {
  for (int c = tid; c < ncols; c += nthreads) {
    const int col = col_base + c;
    float b = 0.f, sc = 1.f;
    if (col < p.c_out) {
      if (p.bias) b = __ldg(p.bias + col);
      if (cbrow) b += __ldg(cbrow + col);
      if (p.out_scale) { sc = __ldg(p.out_scale + col); b = fmaf(sc, b, __ldg(p.out_shift + col)); }
    }
    dst[c] = b;
    if (p.out_scale) dst_scale[c] = sc;
  }
}
__device__ __forceinline__ void epilogue_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ void epilogue_bar_sync256() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
