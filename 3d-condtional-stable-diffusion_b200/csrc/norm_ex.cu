// K6/K7 extended elementwise pass for the VQ-GAN decoder variants (networks/vqgan.py, vqgan_gnorm.py, vqgan_stride.py):
//
//   y[n, vo, c] = post_act( residual[n, vo, c] + act( PReLU_{alpha[vo, c]}( a[n,c] * x[n, src(vo), c] + b[n,c] ) ) )
//
// where (a, b) is a per-channel affine (kind 0) or the GroupNorm affine of (sample, group) statistics (kind 1), and
// src(vo) = vo, or the nearest-neighbour parent voxel when `upsample` is set (layers.UpSampling3D(2): the statistics of the
// up-sampled tensor equal those of the low-resolution one, so GN stats are taken before the replication).
// One HBM pass replaces GroupNormalization -> PReLU -> Add -> ReLU of the residual units (vqgan_gnorm.py:268-286) and
// UpSampling3D -> GroupNormalization -> PReLU of the stride decoder (vqgan_stride.py:447-470).
// Channels-last; C % 8 == 0 runs 16-byte vectors; smaller C (the 1-2 channel network output, fp32) runs per element.
#include "common.cuh"

namespace {

struct ExParams {
  int batch, od, oh, ow, c, kind, groups, act, post_act, upsample, x_f32, y_f32;
  const void* x;
  const float* pa; const float* pb; const float* mean_rstd;
  const act_t* alpha; const act_t* residual;
  void* y;
};

__device__ __forceinline__ int64_t src_voxel(const ExParams& p, int64_t vo) {
  if (!p.upsample) return vo;
  const int w = (int)(vo % p.ow); const int64_t t = vo / p.ow;
  const int h = (int)(t % p.oh), d = (int)(t / p.oh);
  return ((int64_t)(d >> 1) * (p.oh >> 1) + (h >> 1)) * (p.ow >> 1) + (w >> 1);
}

__device__ __forceinline__ void affine_of(const ExParams& p, int n, int c, float& a, float& b) {
  if (p.kind == 0) { a = p.pa[c]; b = p.pb[c]; return; }
  const int g = c / (p.c / p.groups);
  const float m = p.mean_rstd[((int64_t)n * p.groups + g) * 2], r = p.mean_rstd[((int64_t)n * p.groups + g) * 2 + 1];
  a = r * p.pa[c];
  b = p.pb[c] - m * a;
}

// grid = (blocks, batch); C % 8 == 0, bf16 in, bf16 out
__global__ void __launch_bounds__(256) norm_ex_vec_kernel(const ExParams p) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];
  float* sa = sm;
  float* sb = sm + p.c;
  const int n = blockIdx.y;
  for (int c = threadIdx.x; c < p.c; c += blockDim.x) affine_of(p, n, c, sa[c], sb[c]);
  __syncthreads();
  const int c8n = p.c >> 3;
  const int64_t vox_out = (int64_t)p.od * p.oh * p.ow;
  const int64_t vox_in = p.upsample ? vox_out >> 3 : vox_out;
  const int64_t total = vox_out * c8n;
  const act_t* xs = reinterpret_cast<const act_t*>(p.x) + (int64_t)n * vox_in * p.c;
  const act_t* rs = p.residual ? p.residual + (int64_t)n * vox_out * p.c : nullptr;
  act_t* yo = reinterpret_cast<act_t*>(p.y) + (int64_t)n * vox_out * p.c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t vo = i / c8n;
    const int c0 = (int)(i - vo * c8n) << 3;
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(xs + src_voxel(p, vo) * p.c + c0), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], sa[c0 + j], sb[c0 + j]);
    if (p.alpha) {
      float a[8];
      unpack8(*reinterpret_cast<const bf16x8*>(p.alpha + vo * p.c + c0), a);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f) + a[j] * fminf(f[j], 0.f);
    }
    if (p.act != B200DM_ACT_NONE) {
      apply_act_vec(f, p.act);
    }
    if (rs) {
      float r[8];
      unpack8(*reinterpret_cast<const bf16x8*>(rs + vo * p.c + c0), r);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] += r[j];
    }
    if (p.post_act != B200DM_ACT_NONE) {
      apply_act_vec(f, p.post_act);
    }
    *reinterpret_cast<bf16x8*>(yo + vo * p.c + c0) = pack8(f);
  }
}

// per-element path: any C, fp32 or bf16 in / out (network output tensors with 1-2 channels)
__global__ void __launch_bounds__(256) norm_ex_scalar_kernel(const ExParams p) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = blockIdx.y;
  const int64_t vox_out = (int64_t)p.od * p.oh * p.ow;
  const int64_t vox_in = p.upsample ? vox_out >> 3 : vox_out;
  const int64_t total = vox_out * p.c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t vo = i / p.c;
    const int c = (int)(i - vo * p.c);
    const int64_t si = ((int64_t)n * vox_in + src_voxel(p, vo)) * p.c + c;
    float v = p.x_f32 ? reinterpret_cast<const float*>(p.x)[si] : act_to_float(reinterpret_cast<const act_t*>(p.x)[si]);
    float a, b;
    affine_of(p, n, c, a, b);
    v = fmaf(v, a, b);
    if (p.alpha) { const float al = act_to_float(p.alpha[vo * p.c + c]); v = fmaxf(v, 0.f) + al * fminf(v, 0.f); }
    v = apply_act(v, p.act);
    const int64_t oi = ((int64_t)n * vox_out + vo) * p.c + c;
    if (p.residual) v += act_to_float(p.residual[oi]);
    v = apply_act(v, p.post_act);
    if (p.y_f32) reinterpret_cast<float*>(p.y)[oi] = v;
    else reinterpret_cast<act_t*>(p.y)[oi] = float_to_act(v);
  }
}

// whole-sample statistics of an fp32 tensor (GroupNormalization with ONE group on the 1-2 channel network output):
// deterministic two-stage reduction, fp64 combine.  grid = (chunks, batch)
__global__ void __launch_bounds__(256) stats_f32_partial_kernel(const float* __restrict__ x, int64_t per_sample, int chunks,
                                                                double* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = blockIdx.y, ch = blockIdx.x;
  const float* xs = x + (int64_t)n * per_sample;
  const int64_t lo = per_sample * ch / chunks, hi = per_sample * (ch + 1) / chunks;
  double s = 0.0, ss = 0.0;
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) { const double v = xs[i]; s += v; ss += v * v; }
  __shared__ double sh[2][256];
  sh[0][threadIdx.x] = s; sh[1][threadIdx.x] = ss;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { sh[0][threadIdx.x] += sh[0][threadIdx.x + o]; sh[1][threadIdx.x] += sh[1][threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { partial[((int64_t)n * chunks + ch) * 2] = sh[0][0]; partial[((int64_t)n * chunks + ch) * 2 + 1] = sh[1][0]; }
}
__global__ void stats_f32_final_kernel(const double* __restrict__ partial, int batch, int chunks, double count, float eps,
                                       float* __restrict__ mean_rstd) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= batch) return;
  double s = 0.0, ss = 0.0;
  for (int c = 0; c < chunks; ++c) { s += partial[((int64_t)n * chunks + c) * 2]; ss += partial[((int64_t)n * chunks + c) * 2 + 1]; }
  const double m = s / count;
  double var = ss / count - m * m;
  if (var < 0) var = 0;
  mean_rstd[n * 2] = (float)m;
  mean_rstd[n * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
}

constexpr int kStatChunks = 128;

}  // namespace

static int check_ex(const b200dm_norm_ex_desc* d, const char* who) {
  B2_CHECK_ARG(d, "%s: null desc", who);
  B2_CHECK_ARG(d->batch > 0 && d->out_d > 0 && d->out_h > 0 && d->out_w > 0 && d->c > 0, "%s: empty tensor", who);
  B2_CHECK_ARG(d->kind == 0 || (d->kind == 1 && d->groups > 0 && d->c % d->groups == 0), "%s: bad norm kind / groups", who);
  B2_CHECK_ARG(!d->upsample || (d->out_d % 2 == 0 && d->out_h % 2 == 0 && d->out_w % 2 == 0), "%s: upsample needs even output dims", who);
  return B200DM_OK;
}

int bind_norm_act_ex(const b200dm_norm_ex_desc* d, const void* x, const float* a, const float* b, const float* mean_rstd,
                     const void* prelu_alpha, const void* residual, void* y, BoundOp* op) {
  int rc = check_ex(d, "norm_act_ex");
  if (rc) return rc;
  B2_CHECK_ARG(x && a && b && y, "norm_act_ex: null pointer");
  B2_CHECK_ARG(d->kind == 0 || mean_rstd, "norm_act_ex: group norm needs mean_rstd");
  ExParams p;
  p.batch = d->batch; p.od = d->out_d; p.oh = d->out_h; p.ow = d->out_w; p.c = d->c; p.kind = d->kind; p.groups = d->groups;
  p.act = d->act; p.post_act = d->post_act; p.upsample = d->upsample; p.x_f32 = d->x_dtype == B200DM_F32; p.y_f32 = d->y_dtype == B200DM_F32;
  p.x = x; p.pa = a; p.pb = b; p.mean_rstd = mean_rstd; p.alpha = (const act_t*)prelu_alpha;
  p.residual = (const act_t*)residual; p.y = y;
  const int64_t vox = (int64_t)d->out_d * d->out_h * d->out_w;
  const bool vec = d->c % 8 == 0 && !p.x_f32 && !p.y_f32;
  const int64_t items = vec ? vox * (d->c >> 3) : vox * d->c;
  int64_t want = (items * d->batch + 255) / 256;
  const int64_t cap = (int64_t)b2_num_sms() * 8;
  int gx = (int)((want < cap ? want : cap) / d->batch);
  if (gx < 1) gx = 1;
  if (vec) bind_launch(op, norm_ex_vec_kernel, dim3(gx, d->batch), dim3(256), 2 * d->c * sizeof(float), p);
  else bind_launch(op, norm_ex_scalar_kernel, dim3(gx, d->batch), dim3(256), 0, p);
  return B200DM_OK;
}

extern "C" int b200dm_norm_act_ex(const b200dm_norm_ex_desc* d, const void* x, const float* a, const float* b,
                                  const float* mean_rstd, const void* prelu_alpha, const void* residual, void* y, void* stream) {
  return bind_and_run(bind_norm_act_ex, stream, d, x, a, b, mean_rstd, prelu_alpha, residual, y);
}

extern "C" size_t b200dm_stats_f32_workspace(int32_t batch) { return (size_t)batch * kStatChunks * 2 * sizeof(double); }

int bind_stats_f32(const float* x, int32_t batch, int64_t per_sample, float eps, float* mean_rstd, void* workspace,
                   size_t ws_bytes, BoundOp* op) {
  B2_CHECK_ARG(x && mean_rstd && workspace && batch > 0 && per_sample > 0, "stats_f32: bad argument");
  B2_CHECK_ARG(ws_bytes >= b200dm_stats_f32_workspace(batch), "stats_f32: workspace too small");
  bind_launch(op, stats_f32_partial_kernel, dim3(kStatChunks, batch), dim3(256), 0, x, per_sample, kStatChunks, (double*)workspace);
  bind_launch(op, stats_f32_final_kernel, dim3((batch + 63) / 64), dim3(64), 0, (const double*)workspace, batch, kStatChunks,
                  (double)per_sample, eps, mean_rstd);
  return B200DM_OK;
}

extern "C" int b200dm_stats_f32(const float* x, int32_t batch, int64_t per_sample, float eps, float* mean_rstd, void* workspace,
                                size_t ws_bytes, void* stream) {
  return bind_and_run(bind_stats_f32, stream, x, batch, per_sample, eps, mean_rstd, workspace, ws_bytes);
}
