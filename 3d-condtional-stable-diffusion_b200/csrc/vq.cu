// K11: VQ nearest-code search + embedding gather (+ usage histogram) as a shared-memory-tiled
// distance kernel.  d = (||x||^2 + ||e||^2) - 2 x.e in fp32 exactly as VectorQuantizer.get_code_indices
// writes it (networks/vqvae3d_monai.py:165-177), argmin with the lowest index on ties, then the
// gather q = E[idx] (the one_hot @ E^T / embedding_lookup of :139-144, vqgan_attn_cp.py:215).
// fp32 SIMT on purpose: the ranking must be reproducible to the last bit (bf16/TF32 tensor-core
// products flip near-ties); 128x128 block tile, 8x8 register tile, the (N,K) distance matrix
// never leaves the SM.
#include "common.cuh"
#include "vq_tc.cuh"
#include <stdlib.h>

int* b200dm_dbg_flag_ptr();

namespace {

constexpr int BM = 128, BN = 128, BK = 16, PAD = 4;

__global__ void sqnorm_kernel(const float* __restrict__ e, int K, int D, float* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  float s = 0.f;
  for (int d = 0; d < D; ++d) s = __fadd_rn(s, __fmul_rn(e[(int64_t)k * D + d], e[(int64_t)k * D + d]));
  out[k] = s;
}

// Two independent IEEE fp32 FMAs in one issue slot (FFMA2, sm_100): each half rounds exactly like fmaf, so distances and
// indices are bit-identical to the scalar loop; the kernel was issue-bound (76 % issue-active, 81 % of it FFMA).
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void ffma2(uint64_t& acc, uint64_t a, uint64_t b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}

template <bool kBf16>
__device__ __forceinline__ float4 load_x4(const void* x, int64_t row, int D, int d, int64_t N) {
  if (row >= N || d >= D) return make_float4(0.f, 0.f, 0.f, 0.f);
  if (kBf16) {
    const act2_t* p = reinterpret_cast<const act2_t*>(reinterpret_cast<const act_t*>(x) + row * D + d);
    const float2 a = act2_to_float2(p[0]), b = act2_to_float2(p[1]);
    return make_float4(a.x, a.y, b.x, b.y);
  }
  return __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + row * D + d));
}

template <bool kBf16>
__global__ void __launch_bounds__(256, 2) vq_kernel(b200dm_vq_desc dsc, const void* __restrict__ x,
                                                 const float* __restrict__ cb, const float* __restrict__ esq,
                                                 int64_t* __restrict__ idx_out, void* __restrict__ q_out,
                                                 int32_t* __restrict__ hist) {
  // operand tiles, double-buffered: the global loads of tile it+1 are in flight while tile it is multiplied, one
  // __syncthreads per tile.  The cross-thread argmin scratch (rbest / ribest) reuses the tile storage after the main loop.
  constexpr int kTileFloats = BK * (BM + PAD);
  __shared__ __align__(16) float tiles[4 * kTileFloats];   // [buf][X | E][BK][BM + PAD]
  __shared__ float xsq_s[BM];
  __shared__ int final_idx[BM];
  static_assert(4 * kTileFloats >= 2 * BM * 17, "argmin scratch fits in the tile storage");
  float (*rbest)[17] = reinterpret_cast<float (*)[17]>(tiles);
  int (*ribest)[17] = reinterpret_cast<int (*)[17]>(tiles + BM * 17);

  const int D = dsc.d, K = dsc.k;
  const int64_t N = dsc.n;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * BM;

  // ||x||^2 per row, sequential fp32 (2 threads per row would reorder the sum: keep one thread per row)
  if (tid < BM) {
    const int64_t r = row0 + tid;
    float s = 0.f;
    if (r < N) {
      for (int d = 0; d < D; d += 4) {
        const float4 v = load_x4<kBf16>(x, r, D, d, N);
        s = __fadd_rn(s, __fmul_rn(v.x, v.x)); s = __fadd_rn(s, __fmul_rn(v.y, v.y));
        s = __fadd_rn(s, __fmul_rn(v.z, v.z)); s = __fadd_rn(s, __fmul_rn(v.w, v.w));
      }
    }
    xsq_s[tid] = s;
  }

  float best[8];
  int besti[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { best[i] = INFINITY; besti[i] = 0x7fffffff; }

  const int lrow = tid >> 2, ld = (tid & 3) << 2;  // loader: rows lrow, lrow+64; 4 consecutive d
  const int nd = (D + BK - 1) / BK, total = ((K + BN - 1) / BN) * nd;
  float4 xa, xb, ea, eb;
  auto gload = [&](int n0, int d0) {
    xa = load_x4<kBf16>(x, row0 + lrow, D, d0 + ld, N);
    xb = load_x4<kBf16>(x, row0 + lrow + 64, D, d0 + ld, N);
    ea = (n0 + lrow < K && d0 + ld < D) ? __ldg(reinterpret_cast<const float4*>(cb + (int64_t)(n0 + lrow) * D + d0 + ld)) : make_float4(0, 0, 0, 0);
    eb = (n0 + lrow + 64 < K && d0 + ld < D) ? __ldg(reinterpret_cast<const float4*>(cb + (int64_t)(n0 + lrow + 64) * D + d0 + ld)) : make_float4(0, 0, 0, 0);
  };
  auto sstore = [&](int buf) {
    float (*Xs)[BM + PAD] = reinterpret_cast<float (*)[BM + PAD]>(tiles + (2 * buf) * kTileFloats);
    float (*Es)[BN + PAD] = reinterpret_cast<float (*)[BN + PAD]>(tiles + (2 * buf + 1) * kTileFloats);
    Xs[ld + 0][lrow] = xa.x; Xs[ld + 1][lrow] = xa.y; Xs[ld + 2][lrow] = xa.z; Xs[ld + 3][lrow] = xa.w;
    Xs[ld + 0][lrow + 64] = xb.x; Xs[ld + 1][lrow + 64] = xb.y; Xs[ld + 2][lrow + 64] = xb.z; Xs[ld + 3][lrow + 64] = xb.w;
    Es[ld + 0][lrow] = ea.x; Es[ld + 1][lrow] = ea.y; Es[ld + 2][lrow] = ea.z; Es[ld + 3][lrow] = ea.w;
    Es[ld + 0][lrow + 64] = eb.x; Es[ld + 1][lrow + 64] = eb.y; Es[ld + 2][lrow + 64] = eb.z; Es[ld + 3][lrow + 64] = eb.w;
  };
  gload(0, 0);
  sstore(0);
  __syncthreads();   // (also publishes xsq_s)

  uint64_t acc2[8][4];   // acc2[i][jj] = (acc[i][2 jj], acc[i][2 jj + 1])
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) acc2[i][jj] = 0ull;
  int n0 = 0, dt = 0;   // code tile / d tile of iteration `it`
  for (int it = 0; it < total; ++it) {
    const int buf = it & 1;
    const bool more = it + 1 < total;
    const bool last_d = dt + 1 == nd;
    if (more) gload(last_d ? n0 + BN : n0, last_d ? 0 : (dt + 1) * BK);
    {
      const float (*Xs)[BM + PAD] = reinterpret_cast<const float (*)[BM + PAD]>(tiles + (2 * buf) * kTileFloats);
      const float (*Es)[BN + PAD] = reinterpret_cast<const float (*)[BN + PAD]>(tiles + (2 * buf + 1) * kTileFloats);
#pragma unroll
      for (int k = 0; k < BK; ++k) {   // ascending d: the fp32 FMA chain of every (row, code) pair is one fixed sequence
        float a[8], b[8];
        *reinterpret_cast<float4*>(&a[0]) = *reinterpret_cast<const float4*>(&Xs[k][ty * 4]);
        *reinterpret_cast<float4*>(&a[4]) = *reinterpret_cast<const float4*>(&Xs[k][64 + ty * 4]);
        *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&Es[k][tx * 4]);
        *reinterpret_cast<float4*>(&b[4]) = *reinterpret_cast<const float4*>(&Es[k][64 + tx * 4]);
        uint64_t b2[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) b2[jj] = pack2(b[2 * jj], b[2 * jj + 1]);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint64_t a2 = pack2(a[i], a[i]);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) ffma2(acc2[i][jj], a2, b2[jj]);
        }
      }
    }
    if (more) sstore(buf ^ 1);   // last read at iteration it-1, before that iteration's barrier
    __syncthreads();
    if (last_d) {
      // distances for this code tile; running first-min per row
      float acc[8][8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) unpack2(acc2[i][jj], acc[i][2 * jj], acc[i][2 * jj + 1]);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int code = n0 + ((j < 4) ? tx * 4 + j : 64 + tx * 4 + (j - 4));
        if (code < K) {
          const float e2 = __ldg(esq + code);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = (i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4);
            const float dist = __fsub_rn(__fadd_rn(xsq_s[r], e2), __fmul_rn(2.0f, acc[i][j]));
            if (dist < best[i] || (dist == best[i] && code < besti[i])) { best[i] = dist; besti[i] = code; }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) acc2[i][jj] = 0ull;
      n0 += BN; dt = 0;
    } else {
      ++dt;
    }
  }
  // cross-thread (16 threads share a row) reduction
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = (i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4);
    rbest[r][tx] = best[i];
    ribest[r][tx] = besti[i];
  }
  __syncthreads();
  if (tid < BM) {
    float b = rbest[tid][0];
    int bi = ribest[tid][0];
    for (int t = 1; t < 16; ++t) {
      const float v = rbest[tid][t];
      const int vi = ribest[tid][t];
      if (v < b || (v == b && vi < bi)) { b = v; bi = vi; }
    }
    // a row holding a NaN compares false against everything and keeps the sentinel: report code 0 for it (tf.argmin
    // also returns an in-range index for such rows) instead of indexing the histogram / codebook out of bounds
    if ((unsigned)bi >= (unsigned)K) bi = 0;
    final_idx[tid] = bi;
    const int64_t r = row0 + tid;
    if (r < N) {
      idx_out[r] = (int64_t)bi;
      if (hist) atomicAdd(hist + bi, 1);
    }
  }
  __syncthreads();
  if (q_out) {
    // gather: 128 rows x D, 16-byte vectors, one warp streams one row at a time
    const int warp = tid >> 5, lane = tid & 31;
    for (int r = warp; r < BM; r += 8) {
      const int64_t gr = row0 + r;
      if (gr >= N) break;
      const float* src = cb + (int64_t)final_idx[r] * D;
      for (int d = lane * 4; d < D; d += 128) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(src + d));
        if (dsc.q_dtype == B200DM_F32) {
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(q_out) + gr * D + d) = v;
        } else {
          act2_t* o = reinterpret_cast<act2_t*>(reinterpret_cast<act_t*>(q_out) + gr * D + d);
          o[0] = floats_to_act2(v.x, v.y);
          o[1] = floats_to_act2(v.z, v.w);
        }
      }
    }
  }
}

// get_code_indices(..., distribution=True) (vqvae3d_monai.py:165-177): the (N, K) matrix of squared distances itself, with
// the same fp32 chain as vq_kernel (ascending-d FMA, then (||x||^2 + ||e||^2) - 2 x.e), so argmin(row) == the kernel's index.
// A training-time diagnostic of the reference: one thread per (row, code), 16 rows x 16 codes per block through smem.
template <bool kBf16>
__global__ void __launch_bounds__(256) vq_dist_kernel(b200dm_vq_desc dsc, const void* __restrict__ x, const float* __restrict__ cb,
                                                      const float* __restrict__ esq, float* __restrict__ out) {
  __shared__ float xs[16][65], es[16][65];
  const int D = dsc.d, K = dsc.k;
  const int64_t N = dsc.n, row0 = (int64_t)blockIdx.y * 16;
  const int code0 = blockIdx.x * 16, tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc = 0.f, xsq = 0.f;
  for (int d0 = 0; d0 < D; d0 += 64) {
    for (int i = threadIdx.x; i < 16 * 16; i += 256) {   // 16 rows x 16 float4
      const int r = i >> 4, d = d0 + ((i & 15) << 2);
      const float4 v = load_x4<kBf16>(x, row0 + r, D, d, N);
      xs[r][(i & 15) * 4] = v.x; xs[r][(i & 15) * 4 + 1] = v.y; xs[r][(i & 15) * 4 + 2] = v.z; xs[r][(i & 15) * 4 + 3] = v.w;
      const float4 e = (code0 + r < K && d < D) ? __ldg(reinterpret_cast<const float4*>(cb + (int64_t)(code0 + r) * D + d)) : make_float4(0, 0, 0, 0);
      es[r][(i & 15) * 4] = e.x; es[r][(i & 15) * 4 + 1] = e.y; es[r][(i & 15) * 4 + 2] = e.z; es[r][(i & 15) * 4 + 3] = e.w;
    }
    __syncthreads();
    const int nd = (D - d0) < 64 ? (D - d0) : 64;
    for (int d = 0; d < nd; ++d) {
      acc = fmaf(xs[ty][d], es[tx][d], acc);
      xsq = __fadd_rn(xsq, __fmul_rn(xs[ty][d], xs[ty][d]));
    }
    __syncthreads();
  }
  const int64_t r = row0 + ty;
  const int code = code0 + tx;
  if (r < N && code < K) out[r * K + code] = __fsub_rn(__fadd_rn(xsq, __ldg(esq + code)), __fmul_rn(2.0f, acc));
}

}  // namespace

extern "C" int b200dm_vq_distances(const b200dm_vq_desc* d, const void* x, const float* codebook_kd, const float* code_sqnorm,
                                   float* dist, void* stream) {
  B2_CHECK_ARG(d, "vq_distances: null desc");
  if (d->n == 0) return B200DM_OK;
  B2_CHECK_ARG(x && codebook_kd && code_sqnorm && dist, "vq_distances: null argument");
  B2_CHECK_ARG(d->n > 0 && d->k > 0 && d->d > 0 && d->d % 4 == 0, "vq_distances: need d %% 4 == 0, k > 0");
  B2_CHECK_ARG(d->x_dtype == B200DM_F32 || d->x_dtype == B200DM_BF16, "vq_distances: bad x dtype");
  const int64_t by = (d->n + 15) / 16;
  B2_CHECK_ARG(by <= 65535 * 16, "vq_distances: too many rows for one call (diagnostic path; split the input)");
  cudaStream_t s = (cudaStream_t)stream;
  for (int64_t y0 = 0; y0 < by; y0 += 65535) {   // grid.y limit
    const unsigned ny = (unsigned)((by - y0) < 65535 ? (by - y0) : 65535);
    b200dm_vq_desc dd = *d;
    dd.n = d->n - y0 * 16;
    const char* xp = (const char*)x + (size_t)y0 * 16 * d->d * (d->x_dtype == B200DM_F32 ? 4 : 2);
    const dim3 grid((d->k + 15) / 16, ny);
    if (d->x_dtype == B200DM_BF16) vq_dist_kernel<true><<<grid, 256, 0, s>>>(dd, xp, codebook_kd, code_sqnorm, dist + y0 * 16 * d->k);
    else vq_dist_kernel<false><<<grid, 256, 0, s>>>(dd, xp, codebook_kd, code_sqnorm, dist + y0 * 16 * d->k);
  }
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

extern "C" int b200dm_vq_prepare(const float* codebook_kd, int32_t k, int32_t d, float* code_sqnorm, void* stream) {
  B2_CHECK_ARG(codebook_kd && code_sqnorm && k > 0 && d > 0, "vq_prepare: bad arguments");
  sqnorm_kernel<<<(k + 127) / 128, 128, 0, (cudaStream_t)stream>>>(codebook_kd, k, d, code_sqnorm);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

extern "C" int b200dm_vq_argmin_gather(const b200dm_vq_desc* d, const void* x, const float* codebook_kd,
                                       const float* code_sqnorm, int64_t* idx, void* q, int32_t* hist, void* stream) {
  B2_CHECK_ARG(d, "vq_argmin_gather: null desc");
  if (d->n == 0) return B200DM_OK;  // empty input: nothing to do (tf.argmin on (0,K) returns (0,))
  B2_CHECK_ARG(x && codebook_kd && code_sqnorm && idx, "vq_argmin_gather: null argument");
  B2_CHECK_ARG(d->n > 0 && d->k > 0 && d->d > 0 && d->d % 4 == 0 && d->d <= 4096, "vq_argmin_gather: need d %% 4 == 0, 0 < d <= 4096, k > 0");
  B2_CHECK_ARG(d->x_dtype == B200DM_F32 || d->x_dtype == B200DM_BF16, "vq_argmin_gather: bad x dtype");
  B2_CHECK_ARG(d->q_dtype == B200DM_F32 || d->q_dtype == B200DM_BF16, "vq_argmin_gather: bad q dtype");
  const int64_t blocks = (d->n + BM - 1) / BM;
  B2_CHECK_ARG(blocks <= 0x7fffffff, "vq_argmin_gather: too many rows");
  cudaStream_t s = (cudaStream_t)stream;
  if (d->x_dtype == B200DM_BF16)
    vq_kernel<true><<<(unsigned)blocks, 256, 0, s>>>(*d, x, codebook_kd, code_sqnorm, idx, q, hist);
  else
    vq_kernel<false><<<(unsigned)blocks, 256, 0, s>>>(*d, x, codebook_kd, code_sqnorm, idx, q, hist);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

// ---- tensor-core candidate search + exact recheck (vq_tc.cuh): same indices as vq_kernel, bit for bit ----------------------
namespace {

size_t vq_tc_smem_bytes(int k, int d) {
  const int dc = d / 64;
  return 1024 + (size_t)(2 * dc + vqtc::kNSB) * vqtc::kTile + (size_t)k * 4 + 128 * 4 * 2 + (size_t)256 * vqtc::kCap * 8 + 256 * 8 + 128 * 4 +
         (2 * vqtc::kNSB + 4) * 8 + 16;
}
bool vq_tc_supported(int k, int d) {
  return k >= 128 && k % 128 == 0 && d >= 64 && d % 64 == 0 && d <= 256 && vq_tc_smem_bytes(k, d) <= kMaxDynamicSmem;
}
// workspace: [e_hi K*D fp16][e_lo K*D fp16][meta 4 fp32]
size_t vq_tc_ws_bytes(int k, int d) { return (size_t)k * d * 4 + 16; }

}  // namespace

extern "C" size_t b200dm_vq_tc_workspace_bytes(int32_t k, int32_t d) { return vq_tc_supported(k, d) ? vq_tc_ws_bytes(k, d) : 0; }

extern "C" int b200dm_vq_prepare_tc(const float* codebook_kd, const float* code_sqnorm, int32_t k, int32_t d, void* tc_ws, void* stream) {
  B2_CHECK_ARG(codebook_kd && code_sqnorm && tc_ws, "vq_prepare_tc: null argument");
  B2_CHECK_ARG(vq_tc_supported(k, d), "vq_prepare_tc: shape not supported by the tensor-core search (need k %% 128 == 0, d in {64,128,192,256})");
  B2_CHECK_ARG((reinterpret_cast<uintptr_t>(tc_ws) & 127) == 0, "vq_prepare_tc: workspace must be 128-byte aligned");
  __half* ehi = reinterpret_cast<__half*>(tc_ws);
  __half* elo = ehi + (size_t)k * d;
  float* meta = reinterpret_cast<float*>(elo + (size_t)k * d);
  vqtc::vq_tc_prepare_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(codebook_kd, code_sqnorm, k, d, ehi, elo, meta);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

extern "C" int b200dm_vq_argmin_gather_tc(const b200dm_vq_desc* d, const void* x, const float* codebook_kd, const float* code_sqnorm,
                                          const void* tc_ws, int64_t* idx, void* q, int32_t* hist, uint64_t* stats, void* stream) {
  B2_CHECK_ARG(d, "vq_argmin_gather_tc: null desc");
  if (d->n == 0) return B200DM_OK;
  B2_CHECK_ARG(x && codebook_kd && code_sqnorm && tc_ws && idx, "vq_argmin_gather_tc: null argument");
  B2_CHECK_ARG(d->n > 0 && vq_tc_supported(d->k, d->d), "vq_argmin_gather_tc: shape not supported (b200dm_vq_tc_workspace_bytes() == 0): use b200dm_vq_argmin_gather");
  B2_CHECK_ARG(d->x_dtype == B200DM_F32 || d->x_dtype == B200DM_BF16, "vq_argmin_gather_tc: bad x dtype");
  B2_CHECK_ARG(d->q_dtype == B200DM_F32 || d->q_dtype == B200DM_BF16, "vq_argmin_gather_tc: bad q dtype");
  B2_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "vq_argmin_gather_tc: x must be 16-byte aligned");
  const int64_t blocks = (d->n + 127) / 128;
  B2_CHECK_ARG(blocks <= 0x7fffffff, "vq_argmin_gather_tc: too many rows");
  EncodeTiledFn enc = b2_encode_tiled_fn();
  if (!enc) { b200dm_set_error("vq_argmin_gather_tc: cuTensorMapEncodeTiled unavailable"); return B200DM_ERR_CUDA; }
  CUtensorMap maps[2];
  for (int i = 0; i < 2; ++i) {
    cuuint64_t dims[2] = {(cuuint64_t)d->d, (cuuint64_t)d->k};
    cuuint64_t strides[1] = {(cuuint64_t)d->d * 2};
    cuuint32_t box[2] = {64, 128};
    cuuint32_t es[2] = {1, 1};
    void* base = (char*)const_cast<void*>(tc_ws) + (size_t)i * d->k * d->d * 2;
    CUresult r = enc(&maps[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { b200dm_set_error("vq_argmin_gather_tc: cuTensorMapEncodeTiled failed: %d", (int)r); return B200DM_ERR_CUDA; }
  }
  vqtc::Params p;
  p.n = d->n; p.k = d->k; p.d = d->d; p.x = x; p.x_f32 = d->x_dtype == B200DM_F32; p.q_f32 = d->q_dtype == B200DM_F32;
  p.cb = codebook_kd; p.esq = code_sqnorm;
  p.meta = reinterpret_cast<const float*>((const char*)tc_ws + (size_t)d->k * d->d * 4);
  p.idx = idx; p.q = q; p.hist = hist; p.dbg = b200dm_dbg_flag_ptr();
  p.margin_scale = 1.0f;
  p.wave_ctas = b2_num_sms();
  p.stats = reinterpret_cast<unsigned long long*>(stats);
  {   // test hook (B200DM_TUNING=1 only): shrink the candidate margin to measure the headroom of the error bound
    const char* t = getenv("B200DM_TUNING");
    const char* m = (t && t[0] == '1') ? getenv("B200DM_VQ_MARGIN_SCALE") : nullptr;
    if (m) p.margin_scale = (float)atof(m);
  }
  const size_t smem = vq_tc_smem_bytes(d->k, d->d);
  cudaStream_t s = (cudaStream_t)stream;
  if (d->x_dtype == B200DM_BF16) {
    B2_CHECK_CUDA(cudaFuncSetAttribute(vqtc::vq_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    B2_CHECK_CUDA(b2_launch(vqtc::vq_tc_kernel<true>, dim3((unsigned)blocks), dim3(vqtc::kThreads), smem, s, maps[0], maps[1], p));
  } else {
    B2_CHECK_CUDA(cudaFuncSetAttribute(vqtc::vq_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    B2_CHECK_CUDA(b2_launch(vqtc::vq_tc_kernel<false>, dim3((unsigned)blocks), dim3(vqtc::kThreads), smem, s, maps[0], maps[1], p));
  }
  return B200DM_OK;
}
