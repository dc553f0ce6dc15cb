// K6/K7: fused normalisation + activation (+ channel concat) as ONE vectorised, coalesced HBM pass,
// GroupNorm statistics, LayerNorm (3 affine sets per read), row softmax, dtype casts.
// All bf16 activations are NDHWC; every thread moves 16-byte vectors (8 channels).
#include "common.cuh"

namespace {

// ------------------------------------------------------------------ BN fold
__global__ void bn_fold_kernel(const float* gamma, const float* beta, const float* mean, const float* var, float eps,
                               int c, float* scale, float* shift) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) {
    const float inv = gamma[i] * rsqrtf(var[i] + eps);
    scale[i] = inv;
    shift[i] = beta[i] - mean[i] * inv;
  }
}

// ------------------------------------------------------------------ norm + act (+concat)
// grid = (blocks_x, batch).  Prologue folds the per-(sample,channel) affine (a,b) into smem, then a
// grid-stride loop over (voxel, channel-octet) of this sample: y = act(x*a + b).
// The host sizes gridDim.x * 256 as a multiple of C/8 whenever it can, so a thread keeps ONE channel octet for the whole
// pass: its 16 affine coefficients live in registers and the loop is loads / FMAs / stores with no index division
// (ncu on the generic form: 169 warp instructions per 16-byte vector, issue-bound at 2.3 TB/s).
template <int ACT>
__global__ void __launch_bounds__(256, 4) norm_act_kernel(b200dm_norm_desc d, const act_t* __restrict__ x0,
                                                          const act_t* __restrict__ x1,
                                                          const float* __restrict__ pa, const float* __restrict__ pb,
                                                          const float* __restrict__ mean_rstd,
                                                          act_t* __restrict__ y) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];
  const int C = d.c0 + d.c1;
  float* sa = sm;
  float* sb = sm + C;
  const int n = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    if (d.kind == 0) {
      sa[c] = pa[c];
      sb[c] = pb[c];
    } else {
      const int g = c / (C / d.groups);
      const float m = mean_rstd[((int64_t)n * d.groups + g) * 2], r = mean_rstd[((int64_t)n * d.groups + g) * 2 + 1];
      const float a = r * pa[c];
      sa[c] = a;
      sb[c] = pb[c] - m * a;
    }
  }
  __syncthreads();
  const int c8n = C >> 3, c08 = d.c0 >> 3;
  const int64_t total = d.voxels * c8n;
  const act_t* s0 = x0 + (int64_t)n * d.voxels * d.c0;
  const act_t* s1 = x1 ? x1 + (int64_t)n * d.voxels * d.c1 : nullptr;
  act_t* yo = y + (int64_t)n * d.voxels * C;
  constexpr int U = 4;   // independent 16-byte vectors in flight per thread (loads issued before any use)
  const uint32_t tot32 = (uint32_t)total, stride = gridDim.x * blockDim.x;
  const uint32_t i00 = blockIdx.x * blockDim.x + threadIdx.x;
  if (stride % (uint32_t)c8n == 0) {
    const uint32_t c8 = i00 % (uint32_t)c8n, dv = stride / (uint32_t)c8n, nvox = (uint32_t)d.voxels;
    const float4 a0 = *reinterpret_cast<const float4*>(sa + (c8 << 3)), a1 = *reinterpret_cast<const float4*>(sa + (c8 << 3) + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(sb + (c8 << 3)), b1 = *reinterpret_cast<const float4*>(sb + (c8 << 3) + 4);
    const bool first = (int)c8 < c08;
    const act_t* src = first ? s0 + (c8 << 3) : s1 + ((c8 - c08) << 3);
    const uint32_t sstride = first ? d.c0 : d.c1;
    act_t* dst = yo + (c8 << 3);
    for (uint32_t v = i00 / (uint32_t)c8n; v < nvox; v += dv * U) {
      bf16x8 pk[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (v + u * dv < nvox) pk[u] = ldg_bf16x8(reinterpret_cast<const bf16x8*>(src + (size_t)(v + u * dv) * sstride));
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (v + u * dv >= nvox) break;
        float f[8];
        unpack8(pk[u], f);
        f[0] = apply_act(fmaf(f[0], a0.x, b0.x), ACT); f[1] = apply_act(fmaf(f[1], a0.y, b0.y), ACT);
        f[2] = apply_act(fmaf(f[2], a0.z, b0.z), ACT); f[3] = apply_act(fmaf(f[3], a0.w, b0.w), ACT);
        f[4] = apply_act(fmaf(f[4], a1.x, b1.x), ACT); f[5] = apply_act(fmaf(f[5], a1.y, b1.y), ACT);
        f[6] = apply_act(fmaf(f[6], a1.z, b1.z), ACT); f[7] = apply_act(fmaf(f[7], a1.w, b1.w), ACT);
        *reinterpret_cast<bf16x8*>(dst + (size_t)(v + u * dv) * C) = pack8(f);
      }
    }
    return;
  }
  // generic form (grid not aligned to the channel octets): 32-bit index arithmetic (total < 2^31 vectors per sample is
  // checked on the host)
  for (uint32_t i0 = i00; i0 < tot32; i0 += stride * U) {
    bf16x8 pk[U];
    uint32_t vv[U], cc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t i = i0 + u * stride;
      vv[u] = i / (uint32_t)c8n;
      cc[u] = i - vv[u] * (uint32_t)c8n;
      if (i < tot32)
        pk[u] = ((int)cc[u] < c08) ? *reinterpret_cast<const bf16x8*>(s0 + (int64_t)vv[u] * d.c0 + (cc[u] << 3))
                                   : *reinterpret_cast<const bf16x8*>(s1 + (int64_t)vv[u] * d.c1 + ((cc[u] - c08) << 3));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i0 + u * stride >= tot32) break;
      const int c8 = (int)cc[u];
      float f[8];
      unpack8(pk[u], f);
      const float4 a0 = *reinterpret_cast<const float4*>(sa + (c8 << 3)), a1 = *reinterpret_cast<const float4*>(sa + (c8 << 3) + 4);
      const float4 b0 = *reinterpret_cast<const float4*>(sb + (c8 << 3)), b1 = *reinterpret_cast<const float4*>(sb + (c8 << 3) + 4);
      f[0] = apply_act(fmaf(f[0], a0.x, b0.x), ACT); f[1] = apply_act(fmaf(f[1], a0.y, b0.y), ACT);
      f[2] = apply_act(fmaf(f[2], a0.z, b0.z), ACT); f[3] = apply_act(fmaf(f[3], a0.w, b0.w), ACT);
      f[4] = apply_act(fmaf(f[4], a1.x, b1.x), ACT); f[5] = apply_act(fmaf(f[5], a1.y, b1.y), ACT);
      f[6] = apply_act(fmaf(f[6], a1.z, b1.z), ACT); f[7] = apply_act(fmaf(f[7], a1.w, b1.w), ACT);
      *reinterpret_cast<bf16x8*>(yo + (int64_t)vv[u] * C + (c8 << 3)) = pack8(f);
    }
  }
}

// ------------------------------------------------------------------ GroupNorm statistics (deterministic)
// grid = (chunks, batch).  Thread (row r, octet o) keeps per-channel sum / sumsq for its octet over
// voxels r, r+R, ... of the block's chunk; the block reduces in a fixed order and writes one
// (sum, sumsq) pair per group to partial[n][chunk][g].  gn_final combines chunks in fp64.
// kSums: float sums of x (BatchNorm's first pass, groups == C).
// kCentered: float sums of x - center[c] (BatchNorm's second pass, groups == C; see bn_final_kernel).
// kPivot (GroupNorm): the fp32 sums are of d = x - K_g, K_g the chunk's first value of group g's first channel, so they never
// carry the group's offset; the block writes the fp64 sums of x rebuilt from them, sum x = n K + sum d and
// sum x^2 = n K^2 + 2 K sum d + sum d^2 (products of a 16-bit K and fp32 sums: exact in fp64), into double partial[n][chunk][g][2].
// One-pass fp32 sums of x and x^2 would cancel in var = E[x^2] - E[x]^2 once |mean| >> std (at 150 std in fp16: 4e-3 of rstd).
enum GnSums { kSums, kCentered, kPivot };
template <int kMode>
__global__ void __launch_bounds__(256) gn_partial_kernel(const act_t* __restrict__ x, int64_t voxels, int C,
                                                         int groups, int chunks, void* __restrict__ partial,
                                                         const float* __restrict__ center) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float ssum[256 * 8];
  __shared__ float ssq[256 * 8];
  __shared__ float csum[512], csq[512];
  const int c8n = C >> 3;
  const int rows = blockDim.x / c8n;
  const int o = threadIdx.x % c8n, r = threadIdx.x / c8n;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int64_t per = (voxels + chunks - 1) / chunks;
  const int64_t v0 = chunk * per, v1 = (v0 + per < voxels) ? v0 + per : voxels;
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  const act_t* xs = x + (int64_t)n * voxels * C + (o << 3);
  float k[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) k[i] = kMode == kCentered ? center[(o << 3) + i] : 0.f;
  if (kMode == kPivot && v0 < v1) {
    const int cg = C / groups;
#pragma unroll
    for (int i = 0; i < 8; ++i) k[i] = act_to_float(xs[v0 * C - (o << 3) + ((o << 3) + i) / cg * cg]);
  }
  if (r < rows) {
    if constexpr (kMode == kPivot) {
      // the 8 pivots cost a resident block per SM (48 registers instead of 40): two loads in flight per thread make up for it
      for (int64_t v = v0 + r; v < v1; v += 2 * rows) {
        bf16x8 pk[2];
        pk[0] = *reinterpret_cast<const bf16x8*>(xs + v * C);
        if (v + rows < v1) pk[1] = *reinterpret_cast<const bf16x8*>(xs + (v + rows) * C);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (v + u * rows >= v1) break;
          float f[8];
          unpack8(pk[u], f);
#pragma unroll
          for (int i = 0; i < 8; ++i) { f[i] -= k[i]; s[i] += f[i]; q[i] = fmaf(f[i], f[i], q[i]); }
        }
      }
    } else {
      for (int64_t v = v0 + r; v < v1; v += rows) {
        float f[8];
        unpack8(*reinterpret_cast<const bf16x8*>(xs + v * C), f);
        if (kMode == kCentered) {
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] -= k[i];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) { s[i] += f[i]; q[i] = fmaf(f[i], f[i], q[i]); }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) { ssum[threadIdx.x * 8 + i] = s[i]; ssq[threadIdx.x * 8 + i] = q[i]; }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int rr = 0; rr < rows; ++rr) {
      const int t = rr * c8n + (c >> 3);
      a += ssum[t * 8 + (c & 7)];
      b += ssq[t * 8 + (c & 7)];
    }
    csum[c] = a; csq[c] = b;
  }
  __syncthreads();
  const int cg = C / groups;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int c = g * cg; c < (g + 1) * cg; ++c) { a += csum[c]; b += csq[c]; }
    const int64_t i = ((int64_t)n * chunks + chunk) * groups + g;
    if (kMode == kPivot) {
      const double cnt = v0 < v1 ? (double)(v1 - v0) * cg : 0.0;
      const double K = v0 < v1 ? (double)act_to_float(xs[v0 * C - (o << 3) + g * cg]) : 0.0;
      double* p = static_cast<double*>(partial) + i * 2;
      p[0] = cnt * K + (double)a;
      p[1] = cnt * K * K + 2.0 * K * (double)a + (double)b;
    } else {
      float* p = static_cast<float*>(partial) + i * 2;
      p[0] = a; p[1] = b;
    }
  }
}

__global__ void gn_final_kernel(const double* __restrict__ partial, int batch, int groups, int chunks, double count,
                                float eps, float* __restrict__ mean_rstd) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch * groups) return;
  const int n = i / groups, g = i % groups;
  double a = 0.0, b = 0.0;
  for (int c = 0; c < chunks; ++c) {
    const double* p = partial + (((int64_t)n * chunks + c) * groups + g) * 2;
    a += p[0]; b += p[1];
  }
  const double mean = a / count;
  double var = b / count - mean * mean;
  if (var < 0.0) var = 0.0;
  mean_rstd[i * 2] = (float)mean;
  mean_rstd[i * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
}

// BatchNormalization with batch statistics (training=True): per-channel mean and biased variance over all B*D*H*W rows,
// from gn_partial_kernel's per-chunk float sums with groups == C, combined in fixed chunk order in fp64 (bit-reproducible).
// Two passes over x: pass 1 (scale == nullptr) writes center[c] = mean; pass 2 gets the sums of d = x - center and
// forms var = E[d^2] - E[d]^2 -- the corrected two-pass form, so a channel whose |mean| >> std loses nothing to
// cancellation -- then scale = gamma * rsqrt(var + eps), shift = beta - mean * scale: the coefficients norm_act_kernel
// and the conv epilogue's affine read.
__global__ void bn_final_kernel(const float* __restrict__ partial, int C, int chunks, double count, float eps,
                                float* __restrict__ center, const float* __restrict__ gamma, const float* __restrict__ beta,
                                float* __restrict__ scale, float* __restrict__ shift) {
  pdl_launch_dependents();
  pdl_wait();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double a = 0.0, b = 0.0;
  for (int k = 0; k < chunks; ++k) {
    const float* p = partial + ((int64_t)k * C + c) * 2;
    a += (double)p[0]; b += (double)p[1];
  }
  const double d = a / count;
  if (!scale) { center[c] = (float)d; return; }
  double var = b / count - d * d;
  if (var < 0.0) var = 0.0;
  const double mean = (double)center[c] + d;
  const float sc = (float)((double)gamma[c] / sqrt(var + (double)eps));
  scale[c] = sc;
  shift[c] = (float)((double)beta[c] - mean * (double)sc);
}

constexpr int kBnChunks = 256;

// ------------------------------------------------------------------ LayerNorm over C (one warp per row)
template <int kVecPerLane>
__global__ void __launch_bounds__(256) layernorm_kernel(const act_t* __restrict__ x, int64_t rows, int C,
                                                        float eps, int n_out, const float* g0, const float* b0,
                                                        const float* g1, const float* b1, const float* g2,
                                                        const float* b2, act_t* y0, act_t* y1,
                                                        act_t* y2) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp; row < rows; row += nwarps) {
    float f[kVecPerLane][8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kVecPerLane; ++k) {
      const int c = (k * 32 + lane) << 3;
      if (c < C) {
        unpack8(*reinterpret_cast<const bf16x8*>(x + row * C + c), f[k]);
#pragma unroll
        for (int i = 0; i < 8; ++i) s += f[k][i];
      }
    }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < kVecPerLane; ++k) {
      const int c = (k * 32 + lane) << 3;
      if (c < C) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { const float dlt = f[k][i] - mean; q = fmaf(dlt, dlt, q); }
      }
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
#pragma unroll
    for (int k = 0; k < kVecPerLane; ++k) {
      const int c = (k * 32 + lane) << 3;
      if (c < C) {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[k][i] = (f[k][i] - mean) * rstd;
      }
    }
    for (int o = 0; o < n_out; ++o) {
      const float* g = o == 0 ? g0 : (o == 1 ? g1 : g2);
      const float* b = o == 0 ? b0 : (o == 1 ? b1 : b2);
      act_t* y = o == 0 ? y0 : (o == 1 ? y1 : y2);
#pragma unroll
      for (int k = 0; k < kVecPerLane; ++k) {
        const int c = (k * 32 + lane) << 3;
        if (c < C) {
          // affine coefficients as four 16-byte loads (they were 16 scalar loads per output on the row's critical path)
          const float4 ga = __ldg(reinterpret_cast<const float4*>(g + c)), gb = __ldg(reinterpret_cast<const float4*>(g + c + 4));
          const float4 ba = __ldg(reinterpret_cast<const float4*>(b + c)), bb = __ldg(reinterpret_cast<const float4*>(b + c + 4));
          float r[8];
          r[0] = f[k][0] * ga.x + ba.x; r[1] = f[k][1] * ga.y + ba.y; r[2] = f[k][2] * ga.z + ba.z; r[3] = f[k][3] * ga.w + ba.w;
          r[4] = f[k][4] * gb.x + bb.x; r[5] = f[k][5] * gb.y + bb.y; r[6] = f[k][6] * gb.z + bb.z; r[7] = f[k][7] * gb.w + bb.w;
          *reinterpret_cast<bf16x8*>(y + row * C + c) = pack8(r);
        }
      }
    }
  }
}

// ------------------------------------------------------------------ row softmax fp32 -> bf16
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ s, act_t* __restrict__ p,
                                                           int64_t rows, int cols, float scale) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[8];
  __shared__ float bc;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    const float* sr = s + row * cols;
    float m = -INFINITY;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) m = fmaxf(m, sr[c] * scale);
    m = warp_max(m);
    if (lane == 0) red[w] = m;
    __syncthreads();
    if (threadIdx.x == 0) { float t = red[0]; for (int i = 1; i < 8; ++i) t = fmaxf(t, red[i]); bc = t; }
    __syncthreads();
    m = bc;
    float sum = 0.f;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) sum += __expf(sr[c] * scale - m);
    sum = warp_sum(sum);
    __syncthreads();
    if (lane == 0) red[w] = sum;
    __syncthreads();
    if (threadIdx.x == 0) { float t = 0.f; for (int i = 0; i < 8; ++i) t += red[i]; bc = t; }
    __syncthreads();
    const float inv = 1.0f / bc;
    for (int c = threadIdx.x; c < cols; c += blockDim.x)
      p[row * cols + c] = float_to_act(__expf(sr[c] * scale - m) * inv);
    __syncthreads();
  }
}

// ------------------------------------------------------------------ casts
__global__ void __launch_bounds__(256) cast_f32_bf16_kernel(const float* __restrict__ x, act_t* __restrict__ y,
                                                            int64_t n) {
  const int64_t n8 = n >> 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float f[8];
    *reinterpret_cast<float4*>(&f[0]) = __ldg(reinterpret_cast<const float4*>(x + (i << 3)));
    *reinterpret_cast<float4*>(&f[4]) = __ldg(reinterpret_cast<const float4*>(x + (i << 3) + 4));
    *reinterpret_cast<bf16x8*>(y + (i << 3)) = pack8(f);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 7)) y[(n8 << 3) + threadIdx.x] = float_to_act(x[(n8 << 3) + threadIdx.x]);
}
__global__ void __launch_bounds__(256) cast_bf16_f32_kernel(const act_t* __restrict__ x, float* __restrict__ y,
                                                            int64_t n) {
  const int64_t n8 = n >> 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(x + (i << 3)), f);
    *reinterpret_cast<float4*>(y + (i << 3)) = *reinterpret_cast<float4*>(&f[0]);
    *reinterpret_cast<float4*>(y + (i << 3) + 4) = *reinterpret_cast<float4*>(&f[4]);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 7)) y[(n8 << 3) + threadIdx.x] = act_to_float(x[(n8 << 3) + threadIdx.x]);
}

// ------------------------------------------------------------------ small fp32 dense
// y[m][n] = act_out( sum_k act_in(x[m][k]) * w[k][n] + b[n] ).  One thread per output column, 8 rows per block.
__global__ void __launch_bounds__(128) dense_f32_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                        const float* __restrict__ b, float* __restrict__ y, int M, int K,
                                                        int64_t N, int act_in, int act_out) {
  extern __shared__ float xs[];  // [8][K]
  const int m0 = blockIdx.y * 8;
  for (int i = threadIdx.x; i < 8 * K; i += blockDim.x) {
    const int r = i / K, k = i - r * K;
    float v = (m0 + r < M) ? x[(int64_t)(m0 + r) * K + k] : 0.f;
    if (act_in == B200DM_ACT_SILU) v = v / (1.0f + expf(-v));
    xs[i] = v;
  }
  __syncthreads();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float acc[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) acc[r] = 0.f;
  for (int k = 0; k < K; ++k) {
    const float wv = __ldg(w + (int64_t)k * N + n);
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r] = fmaf(xs[r * K + k], wv, acc[r]);
  }
  const float bias = b ? b[n] : 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    if (m0 + r < M) {
      float v = acc[r] + bias;
      if (act_out == B200DM_ACT_SILU) v = v / (1.0f + expf(-v));
      else if (act_out == B200DM_ACT_RELU) v = fmaxf(v, 0.f);
      y[(int64_t)(m0 + r) * N + n] = v;
    }
  }
}

inline int grid_for(int64_t work_items, int threads, int waves = 8) {
  const int64_t want = (work_items + threads - 1) / threads;
  const int64_t cap = (int64_t)b2_num_sms() * waves;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace

extern "C" int b200dm_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, float eps,
                              int32_t c, float* scale, float* shift, void* stream) {
  B2_CHECK_ARG(gamma && beta && mean && var && scale && shift && c > 0, "bn_fold: bad arguments");
  bn_fold_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(gamma, beta, mean, var, eps, c, scale, shift);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

static int check_norm_desc(const b200dm_norm_desc* d, const char* who) {
  B2_CHECK_ARG(d, "%s: null desc", who);
  const int C = d->c0 + d->c1;
  B2_CHECK_ARG(d->voxels > 0 && d->batch > 0, "%s: empty tensor", who);
  B2_CHECK_ARG(d->c0 > 0 && d->c0 % 8 == 0 && d->c1 >= 0 && d->c1 % 8 == 0, "%s: channel counts must be multiples of 8 (got %d,%d)", who, d->c0, d->c1);
  B2_CHECK_ARG(C <= 1024, "%s: C=%d > 1024 unsupported", who, C);
  B2_CHECK_ARG(d->kind == 0 || d->kind == 1, "%s: kind must be 0 or 1", who);
  if (d->kind == 1) B2_CHECK_ARG(d->groups > 0 && C % d->groups == 0, "%s: groups=%d does not divide C=%d", who, d->groups, C);
  B2_CHECK_ARG(d->x_dtype == B200DM_BF16 && d->y_dtype == B200DM_BF16, "%s: only bf16 activations are supported", who);
  B2_CHECK_ARG(d->batch <= 65535, "%s: batch too large", who);
  return B200DM_OK;
}

extern "C" size_t b200dm_gn_stats_workspace(const b200dm_norm_desc* d) {
  if (!d || d->groups <= 0) return 0;
  const int chunks = 64;
  return (size_t)d->batch * chunks * d->groups * 2 * sizeof(double);
}

int bind_gn_stats(const b200dm_norm_desc* d, const void* x, float eps, float* mean_rstd, float* workspace, size_t ws_bytes,
                  BoundOp* op) {
  int rc = check_norm_desc(d, "gn_stats");
  if (rc) return rc;
  B2_CHECK_ARG(d->kind == 1 && d->c1 == 0, "gn_stats: kind must be 1 with a single source");
  B2_CHECK_ARG(x && mean_rstd && workspace, "gn_stats: null pointer");
  B2_CHECK_ARG(((uintptr_t)workspace & 7) == 0, "gn_stats: workspace must be 8-byte aligned");
  B2_CHECK_ARG(ws_bytes >= b200dm_gn_stats_workspace(d), "gn_stats: workspace too small");
  const int C = d->c0;
  B2_CHECK_ARG(C <= 512 && 256 % (C / 8) == 0, "gn_stats: C=%d unsupported (need C/8 to divide 256, C<=512)", C);
  const int chunks = 64;
  bind_launch(op, gn_partial_kernel<kPivot>, dim3(chunks, d->batch), dim3(256), 0, (const act_t*)x, d->voxels, C, d->groups, chunks,
                  (void*)workspace, (const float*)nullptr);
  const int tot = d->batch * d->groups;
  bind_launch(op, gn_final_kernel, dim3((tot + 127) / 128), dim3(128), 0, (const double*)workspace, d->batch, d->groups, chunks,
                  (double)d->voxels * (double)(C / d->groups), eps, mean_rstd);
  return B200DM_OK;
}

extern "C" int b200dm_gn_stats(const b200dm_norm_desc* d, const void* x, float eps, float* mean_rstd, float* workspace,
                               size_t ws_bytes, void* stream) {
  return bind_and_run(bind_gn_stats, stream, d, x, eps, mean_rstd, workspace, ws_bytes);
}

extern "C" size_t b200dm_bn_stats_workspace(int32_t c) {
  return c > 0 ? ((size_t)kBnChunks * c * 2 + c) * sizeof(float) : 0;
}

int bind_bn_stats(const void* x, int64_t rows, int32_t c, const float* gamma, const float* beta, float eps, float* scale,
                  float* shift, float* workspace, size_t ws_bytes, BoundOp* op) {
  B2_CHECK_ARG(x && gamma && beta && scale && shift && workspace && rows > 0, "bn_stats: bad arguments");
  B2_CHECK_ARG(c >= 8 && c <= 512 && c % 8 == 0 && 256 % (c / 8) == 0, "bn_stats: C=%d unsupported (need C/8 to divide 256, 8 <= C <= 512)", c);
  B2_CHECK_ARG(ws_bytes >= b200dm_bn_stats_workspace(c), "bn_stats: workspace too small");
  float* center = workspace + (size_t)kBnChunks * c * 2;
  const act_t* xb = (const act_t*)x;
  const dim3 fgrid((c + 127) / 128);
  bind_launch(op, gn_partial_kernel<kSums>, dim3(kBnChunks), dim3(256), 0, xb, rows, (int)c, (int)c, kBnChunks, (void*)workspace,
                  (const float*)nullptr);
  bind_launch(op, bn_final_kernel, fgrid, dim3(128), 0, (const float*)workspace, (int)c, kBnChunks, (double)rows, eps, center,
                  (const float*)nullptr, (const float*)nullptr, (float*)nullptr, (float*)nullptr);
  bind_launch(op, gn_partial_kernel<kCentered>, dim3(kBnChunks), dim3(256), 0, xb, rows, (int)c, (int)c, kBnChunks, (void*)workspace,
                  (const float*)center);
  bind_launch(op, bn_final_kernel, fgrid, dim3(128), 0, (const float*)workspace, (int)c, kBnChunks, (double)rows, eps, center, gamma, beta,
                  scale, shift);
  return B200DM_OK;
}

extern "C" int b200dm_bn_stats(const void* x, int64_t rows, int32_t c, const float* gamma, const float* beta, float eps,
                               float* scale, float* shift, float* workspace, size_t ws_bytes, void* stream) {
  return bind_and_run(bind_bn_stats, stream, x, rows, c, gamma, beta, eps, scale, shift, workspace, ws_bytes);
}

int bind_norm_act_fwd(const b200dm_norm_desc* d, const void* x0, const void* x1, const float* a, const float* b,
                      const float* mean_rstd, void* y, BoundOp* op) {
  int rc = check_norm_desc(d, "norm_act_fwd");
  if (rc) return rc;
  B2_CHECK_ARG(x0 && a && b && y, "norm_act_fwd: null pointer");
  B2_CHECK_ARG((d->c1 == 0) == (x1 == nullptr), "norm_act_fwd: x1 must be given iff c1 > 0");
  B2_CHECK_ARG(d->kind == 0 || mean_rstd, "norm_act_fwd: group norm needs mean_rstd");
  const int C = d->c0 + d->c1;
  const int64_t items = d->voxels * (C >> 3);
  B2_CHECK_ARG(items < (1ll << 31), "norm_act_fwd: more than 2^31 16-byte vectors per sample");
  // one resident wave (blocks per SM from the occupancy calculator), gridDim.x * 256 a multiple of C/8 when affordable
  static int occ[3] = {0, 0, 0};
  const int ai = d->act == B200DM_ACT_SILU ? 1 : (d->act == B200DM_ACT_RELU ? 2 : 0);
  auto kern = ai == 1 ? norm_act_kernel<B200DM_ACT_SILU> : (ai == 2 ? norm_act_kernel<B200DM_ACT_RELU> : norm_act_kernel<B200DM_ACT_NONE>);
  if (occ[ai] == 0) {
    int o = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, 256, 2 * 512 * sizeof(float)) != cudaSuccess || o < 1) o = 4;
    occ[ai] = o;
  }
  int gx = grid_for((items * d->batch + 3) / 4, 256, occ[ai]);
  gx = (gx + d->batch - 1) / d->batch;
  if (gx < 1) gx = 1;
  {
    const int c8n = C >> 3;
    int g = c8n, r = 256;   // gcd(c8n, 256)
    while (r) { const int t = g % r; g = r; r = t; }
    const int m = c8n / g;   // gridDim.x must be a multiple of m for the fixed-octet path
    if (m > 1 && (int64_t)gx * 256 < items) gx = (gx + m - 1) / m * m;
  }
  bind_launch(op, kern, dim3(gx, d->batch), dim3(256), 2 * C * sizeof(float), *d, (const act_t*)x0, (const act_t*)x1, a, b, mean_rstd,
                  (act_t*)y);
  return B200DM_OK;
}

extern "C" int b200dm_norm_act_fwd(const b200dm_norm_desc* d, const void* x0, const void* x1, const float* a,
                                   const float* b, const float* mean_rstd, void* y, void* stream) {
  return bind_and_run(bind_norm_act_fwd, stream, d, x0, x1, a, b, mean_rstd, y);
}

int bind_layernorm_fwd(const void* x, int64_t rows, int32_t c, float eps, int32_t n_out, const float* const* gammas,
                       const float* const* betas, void* const* ys, BoundOp* op) {
  B2_CHECK_ARG(x && rows > 0 && gammas && betas && ys, "layernorm_fwd: bad arguments");
  B2_CHECK_ARG(c > 0 && c % 8 == 0 && c <= 1024, "layernorm_fwd: C=%d unsupported (multiple of 8, <= 1024)", c);
  B2_CHECK_ARG(n_out >= 1 && n_out <= 3, "layernorm_fwd: n_out must be 1..3");
  const float* g[3] = {nullptr, nullptr, nullptr};
  const float* b[3] = {nullptr, nullptr, nullptr};
  act_t* y[3] = {nullptr, nullptr, nullptr};
  for (int i = 0; i < n_out; ++i) {
    g[i] = gammas[i]; b[i] = betas[i]; y[i] = (act_t*)ys[i];
    B2_CHECK_ARG(g[i] && b[i] && y[i], "layernorm_fwd: null affine/output %d", i);
    B2_CHECK_ARG(((uintptr_t)g[i] & 15) == 0 && ((uintptr_t)b[i] & 15) == 0, "layernorm_fwd: gamma/beta %d must be 16-byte aligned", i);
  }
  const int grid = grid_for(rows * 32, 256, 8);
  auto kern = c <= 256 ? layernorm_kernel<1> : (c <= 512 ? layernorm_kernel<2> : layernorm_kernel<4>);
  bind_launch(op, kern, dim3(grid), dim3(256), 0, (const act_t*)x, rows, c, eps, n_out, g[0], b[0], g[1], b[1], g[2], b[2], y[0], y[1], y[2]);
  return B200DM_OK;
}

extern "C" int b200dm_layernorm_fwd(const void* x, int64_t rows, int32_t c, float eps, int32_t n_out,
                                    const float* const* gammas, const float* const* betas, void* const* ys,
                                    void* stream) {
  return bind_and_run(bind_layernorm_fwd, stream, x, rows, c, eps, n_out, gammas, betas, ys);
}

int bind_softmax_rows(const float* s, void* p_bf16, int64_t rows, int32_t cols, float scale, BoundOp* op) {
  B2_CHECK_ARG(s && p_bf16 && rows > 0 && cols > 0, "softmax_rows: bad arguments");
  const int64_t cap = (int64_t)b2_num_sms() * 8;
  const int grid = (int)(rows < cap ? rows : cap);
  bind_launch(op, softmax_rows_kernel, dim3(grid), dim3(256), 0, s, (act_t*)p_bf16, rows, cols, scale);
  return B200DM_OK;
}

extern "C" int b200dm_softmax_rows(const float* s, void* p_bf16, int64_t rows, int32_t cols, float scale, void* stream) {
  return bind_and_run(bind_softmax_rows, stream, s, p_bf16, rows, cols, scale);
}

extern "C" int b200dm_cast(const void* x, int32_t x_dtype, void* y, int32_t y_dtype, int64_t n, void* stream) {
  B2_CHECK_ARG(x && y && n > 0, "cast: bad arguments");
  const int grid = grid_for((n + 7) / 8, 256, 8);
  cudaStream_t s = (cudaStream_t)stream;
  if (x_dtype == B200DM_F32 && y_dtype == B200DM_BF16) cast_f32_bf16_kernel<<<grid, 256, 0, s>>>((const float*)x, (act_t*)y, n);
  else if (x_dtype == B200DM_BF16 && y_dtype == B200DM_F32) cast_bf16_f32_kernel<<<grid, 256, 0, s>>>((const act_t*)x, (float*)y, n);
  else { b200dm_set_error("cast: unsupported dtype pair %d -> %d", x_dtype, y_dtype); return B200DM_ERR_UNSUPPORTED; }
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

extern "C" int b200dm_dense_f32(const float* x, const float* w, const float* b, float* y, int32_t m, int32_t k,
                                int64_t n, int32_t act_in, int32_t act_out, void* stream) {
  B2_CHECK_ARG(x && w && y && m > 0 && k > 0 && n > 0, "dense_f32: bad arguments");
  B2_CHECK_ARG((size_t)k * 8 * sizeof(float) <= 48 * 1024, "dense_f32: K=%d too large", k);
  B2_CHECK_ARG((m + 7) / 8 <= 65535, "dense_f32: M too large");
  dim3 grid((unsigned)((n + 127) / 128), (unsigned)((m + 7) / 8));
  dense_f32_kernel<<<grid, 128, (size_t)k * 8 * sizeof(float), (cudaStream_t)stream>>>(x, w, b, y, m, k, n, act_in, act_out);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

// out[r][:] = table[idx[r]][:] (fp32): per-sample timestep rows of the hoisted Dense(swish(temb)) tables when the network is
// called with a (B,) vector of DISTINCT timesteps (train_step draws t ~ U{0..T-1} per sample, conditional_dm3d.py:474,493)
namespace {
__global__ void gather_rows_kernel(const float* __restrict__ table, const int32_t* __restrict__ idx, float* __restrict__ out,
                                   int rows, int cols, int table_rows) {
  const int r = blockIdx.y;
  int t = idx[r];
  t = t < 0 ? 0 : (t >= table_rows ? table_rows - 1 : t);
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x)
    out[(int64_t)r * cols + c] = table[(int64_t)t * cols + c];
}
}  // namespace

extern "C" int b200dm_gather_rows_f32(const float* table, int32_t table_rows, const int32_t* idx, float* out, int32_t rows,
                                      int32_t cols, void* stream) {
  B2_CHECK_ARG(table && idx && out && rows > 0 && cols > 0 && table_rows > 0 && rows <= 65535, "gather_rows_f32: bad arguments");
  gather_rows_kernel<<<dim3((cols + 255) / 256, rows), 256, 0, (cudaStream_t)stream>>>(table, idx, out, rows, cols, table_rows);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}
