// K10: fused reverse-diffusion update with an in-register Philox4x32-10 noise stream.
// One HBM pass: read x_t (fp32) + eps (bf16|fp32) [+ injected noise], write x_{t-1} (fp32) [+ bf16 copy
// for the next U-Net input conv].  Replaces ~10 TF elementwise ops + tf.random.normal per step
// (networks/dm3d.py:477-508, 516-530).  Arithmetic follows the reference op by op in fp32
// (__fmul_rn/__fadd_rn/__fdiv_rn forbid FMA contraction so the result matches separate TF ops).
#include "common.cuh"
#include "update_math.cuh"

namespace {

using namespace upd;

constexpr uint32_t kTrainNoiseStream = 2;   // Philox stream id of train_step's noise

// 8 elements per thread per trip (two Philox counters), two trips in flight: 4x LDG.128 x_t, 2-4x LDG.128 eps issued before
// any use; grid = (blocks, batch) so the loop has no index division.
template <bool kEpsBf16>
__global__ void __launch_bounds__(256, 4) update_kernel(b200dm_update_desc d, const float* __restrict__ x_t,
                                                     const void* __restrict__ eps, const float* __restrict__ noise,
                                                     float* __restrict__ x_prev, act_t* __restrict__ x_bf16) {
  pdl_launch_dependents();
  pdl_wait();
  const Coef k = load_coef(d);
  const uint32_t n8 = (uint32_t)(d.n_per_sample >> 3);
  const int64_t b = blockIdx.y, base = b * d.n_per_sample;
  const bool gen = (noise == nullptr) && d.sampler == 0 && k.t > 0;
  const bool inj = noise != nullptr && k.t > 0;
  // reserved bit 0: the Philox key and the global index of sample 0 live in device memory (t_dev[4..7]), so a captured step
  // graph serves every seed / shard without re-capture; desc.sample_id0 is then this launch's offset inside the call's batch
  uint64_t seed = d.seed;
  int64_t sid0 = d.sample_id0;
  if ((d.reserved & 1) && d.t_dev) {
    seed = (uint64_t)(uint32_t)d.t_dev[4] | ((uint64_t)(uint32_t)d.t_dev[5] << 32);
    sid0 += (int64_t)((uint64_t)(uint32_t)d.t_dev[6] | ((uint64_t)(uint32_t)d.t_dev[7] << 32));
  }
  const uint32_t stride = gridDim.x * blockDim.x;
  constexpr int U = 2;
  for (uint32_t j0 = blockIdx.x * blockDim.x + threadIdx.x; j0 < n8; j0 += stride * U) {
    float x[U][8], e[U][8];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t j = j0 + u * stride;
      if (j >= n8) break;
      const int64_t off = base + ((int64_t)j << 3);
      *reinterpret_cast<float4*>(&x[u][0]) = __ldg(reinterpret_cast<const float4*>(x_t + off));
      *reinterpret_cast<float4*>(&x[u][4]) = __ldg(reinterpret_cast<const float4*>(x_t + off + 4));
      if (kEpsBf16) {
        unpack8(ldg_bf16x8(reinterpret_cast<const bf16x8*>(reinterpret_cast<const act_t*>(eps) + off)), e[u]);
      } else {
        *reinterpret_cast<float4*>(&e[u][0]) = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(eps) + off));
        *reinterpret_cast<float4*>(&e[u][4]) = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(eps) + off + 4));
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t j = j0 + u * stride;
      if (j >= n8) break;
      const int64_t off = base + ((int64_t)j << 3);
      float z[8];
      if (gen) {
        float za[4], zb[4];
        normal4(2 * j, (uint32_t)k.t, (uint32_t)(sid0 + b), 0u, seed, za);
        normal4(2 * j + 1, (uint32_t)k.t, (uint32_t)(sid0 + b), 0u, seed, zb);
#pragma unroll
        for (int q = 0; q < 4; ++q) { z[q] = za[q]; z[4 + q] = zb[q]; }
      } else if (inj) {
        *reinterpret_cast<float4*>(&z[0]) = __ldg(reinterpret_cast<const float4*>(noise + off));
        *reinterpret_cast<float4*>(&z[4]) = __ldg(reinterpret_cast<const float4*>(noise + off + 4));
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) z[q] = 0.0f;
      }
      float y[8];
      step_vec(k, d.sampler, x[u], e[u], z, y);
      *reinterpret_cast<float4*>(x_prev + off) = *reinterpret_cast<float4*>(&y[0]);
      *reinterpret_cast<float4*>(x_prev + off + 4) = *reinterpret_cast<float4*>(&y[4]);
      if (x_bf16) *reinterpret_cast<bf16x8*>(x_bf16 + off) = pack8(y);
    }
  }
}

__global__ void __launch_bounds__(256) philox_normal_kernel(float* __restrict__ x, act_t* __restrict__ xb,
                                                            int64_t n_per_sample, int batch, uint64_t seed,
                                                            int64_t sample_id0, int step, int stream_id) {
  const int64_t n4 = n_per_sample >> 2, total = n4 * batch;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n4, j = i - b * n4;
    float z[4];
    normal4((uint32_t)j, (uint32_t)step, (uint32_t)(sample_id0 + b), (uint32_t)stream_id, seed, z);
    const int64_t off = b * n_per_sample + (j << 2);
    *reinterpret_cast<float4*>(x + off) = *reinterpret_cast<float4*>(&z[0]);
    if (xb) {
      *reinterpret_cast<act2_t*>(xb + off) = floats_to_act2(z[0], z[1]);
      *reinterpret_cast<act2_t*>(xb + off + 2) = floats_to_act2(z[2], z[3]);
    }
  }
}

// Forward diffusion of train_step (conditional_dm3d.py:481-490): x_t = sqrt(abar_t) * z + sqrt(1 - abar_t) * noise for a
// per-sample t, in the reference's fp32 op order (two rounded products, one rounded sum).  The noise is Philox stream 2,
// counter (element / 4, 0, global sample index, 2) -- streams 0 (update) and 1 (x_T) belong to the sampler -- or injected.
// grid = (blocks, batch); 4 elements per thread per trip.
__global__ void __launch_bounds__(256) q_sample_kernel(const float* __restrict__ z, const float* __restrict__ sqrt_ab,
                                                       const float* __restrict__ sqrt_1mab, const int32_t* __restrict__ t,
                                                       const float* __restrict__ noise, int64_t n_per_sample, uint64_t seed,
                                                       int64_t sample_id0, act_t* __restrict__ x16, float* __restrict__ x32) {
  pdl_launch_dependents();
  pdl_wait();
  const int64_t b = blockIdx.y, base = b * n_per_sample;
  const int tb = t[b];
  const float a = sqrt_ab[tb], s = sqrt_1mab[tb];
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < (n_per_sample >> 2); j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t off = base + (j << 2);
    float x[4], e[4];
    *reinterpret_cast<float4*>(x) = __ldg(reinterpret_cast<const float4*>(z + off));
    if (noise) *reinterpret_cast<float4*>(e) = __ldg(reinterpret_cast<const float4*>(noise + off));
    else normal4((uint32_t)j, 0u, (uint32_t)(sample_id0 + b), kTrainNoiseStream, seed, e);
#pragma unroll
    for (int q = 0; q < 4; ++q) x[q] = __fadd_rn(__fmul_rn(a, x[q]), __fmul_rn(s, e[q]));
    *reinterpret_cast<act2_t*>(x16 + off) = floats_to_act2(x[0], x[1]);
    *reinterpret_cast<act2_t*>(x16 + off + 2) = floats_to_act2(x[2], x[3]);
    if (x32) *reinterpret_cast<float4*>(x32 + off) = *reinterpret_cast<float4*>(x);
  }
}

// sum over all elements of (noise - eps_hat)^2, per block in fixed order (fp64), one partial per block: the numerator of
// train_step's MSE(reduction=SUM) (conditional_dm3d.py:496-499).  The noise is regenerated from q_sample_kernel's stream (or
// read when injected).  grid = (blocks, batch)
constexpr int kLossBlocks = 64;
__global__ void __launch_bounds__(256) sq_err_partial_kernel(const float* __restrict__ eps, const float* __restrict__ noise,
                                                             int64_t n_per_sample, uint64_t seed, int64_t sample_id0,
                                                             double* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  const int64_t b = blockIdx.y, base = b * n_per_sample;
  double acc = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < (n_per_sample >> 2); j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t off = base + (j << 2);
    float y[4], e[4];
    *reinterpret_cast<float4*>(y) = __ldg(reinterpret_cast<const float4*>(eps + off));
    if (noise) *reinterpret_cast<float4*>(e) = __ldg(reinterpret_cast<const float4*>(noise + off));
    else normal4((uint32_t)j, 0u, (uint32_t)(sample_id0 + b), kTrainNoiseStream, seed, e);
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) { const float d = __fsub_rn(e[q], y[q]); s = __fadd_rn(s, __fmul_rn(d, d)); }
    acc += (double)s;
  }
  __shared__ double red[256];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[b * gridDim.x + blockIdx.x] = red[0];
}

__global__ void sq_err_final_kernel(const double* __restrict__ partial, int n, double inv_divisor, float* __restrict__ loss) {
  pdl_launch_dependents();
  pdl_wait();
  double a = 0.0;
  for (int i = 0; i < n; ++i) a += partial[i];
  *loss = (float)(a * inv_divisor);
}

__global__ void step_advance_kernel(int32_t* t_dev, int32_t delta) {
  pdl_launch_dependents();
  pdl_wait();
  t_dev[0] += delta;
  t_dev[1] += delta;
}

// t_dev = [t, t_prev, idx, -]: move to the next entry of a device-resident timestep sequence (terminated by -1), so one
// captured step graph replays ANY sequence -- every DDPM range, strided DDIM, non-uniform spacings -- with no host work.
__global__ void step_advance_seq_kernel(int32_t* t_dev, const int32_t* __restrict__ seq) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = t_dev[2] + 1;
  t_dev[2] = i;
  const int t = seq[i];
  t_dev[0] = t < 0 ? 0 : t;                 // past the end: stay on a valid table row (the step's result is unused)
  t_dev[1] = t < 0 ? -1 : seq[i + 1];
}

}  // namespace

int bind_ddpm_update(const b200dm_update_desc* d, const float* x_t, const void* eps, const float* noise, float* x_prev,
                     void* x_prev_bf16, BoundOp* op) {
  B2_CHECK_ARG(d && x_t && eps && x_prev, "ddpm_update: null argument");
  B2_CHECK_ARG(d->n_per_sample > 0 && d->n_per_sample % 8 == 0, "ddpm_update: n_per_sample must be a positive multiple of 8");
  B2_CHECK_ARG(d->batch > 0, "ddpm_update: batch must be > 0");
  B2_CHECK_ARG(d->sampler == 0 || d->sampler == 1, "ddpm_update: sampler must be 0 (ddpm) or 1 (ddim)");
  B2_CHECK_ARG(d->beta && d->sqrt_alpha && d->alpha_bar && d->alpha_bar_prev && d->sqrt_alpha_bar &&
                   d->sqrt_alpha_bar_prev && d->sqrt_one_minus_alpha_bar, "ddpm_update: null schedule table");
  B2_CHECK_ARG(d->t_dev || d->t >= 0, "ddpm_update: negative timestep");
  B2_CHECK_ARG((d->n_per_sample >> 3) < (1ll << 31) && d->batch <= 65535, "ddpm_update: sample too large / batch > 65535");
  const int64_t per = (d->n_per_sample >> 3), want = (per + 2 * 256 - 1) / (2 * 256);
  int64_t cap = ((int64_t)b2_num_sms() * 4 + d->batch - 1) / d->batch;   // one resident wave: 4 blocks per SM (62 registers)
  if (cap < 1) cap = 1;
  const dim3 grid((unsigned)(want < cap ? want : cap), (unsigned)d->batch);
  bind_launch(op, d->eps_dtype == B200DM_BF16 ? update_kernel<true> : update_kernel<false>, grid, dim3(256), 0, *d, x_t, eps, noise, x_prev,
                  (act_t*)x_prev_bf16);
  return B200DM_OK;
}

extern "C" int b200dm_ddpm_update(const b200dm_update_desc* d, const float* x_t, const void* eps,
                                  const float* noise, float* x_prev, void* x_prev_bf16, void* stream) {
  return bind_and_run(bind_ddpm_update, stream, d, x_t, eps, noise, x_prev, x_prev_bf16);
}

extern "C" int b200dm_philox_normal(float* x, void* x_bf16, int64_t n_per_sample, int32_t batch, uint64_t seed,
                                    int64_t sample_id0, int32_t step, int32_t stream_id, void* stream) {
  B2_CHECK_ARG(x && n_per_sample > 0 && n_per_sample % 4 == 0 && batch > 0, "philox_normal: bad arguments");
  const int64_t total = (n_per_sample >> 2) * batch;
  const int64_t want = (total + 255) / 256;
  const int grid = (int)(want < (int64_t)b2_num_sms() * 8 ? want : (int64_t)b2_num_sms() * 8);
  philox_normal_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, (act_t*)x_bf16, n_per_sample, batch, seed,
                                                              sample_id0, step, stream_id);
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

extern "C" int b200dm_step_advance_seq(int32_t* t_dev, const int32_t* seq, void* stream) {
  B2_CHECK_ARG(t_dev && seq, "step_advance_seq: null argument");
  B2_CHECK_CUDA(b2_launch(step_advance_seq_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, t_dev, seq));
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

int bind_step_advance(int32_t* t_dev, int32_t delta, BoundOp* op) {
  B2_CHECK_ARG(t_dev, "step_advance: null t_dev");
  bind_launch(op, step_advance_kernel, dim3(1), dim3(1), 0, t_dev, delta);
  return B200DM_OK;
}

extern "C" int b200dm_step_advance(int32_t* t_dev, int32_t delta, void* stream) {
  return bind_and_run(bind_step_advance, stream, t_dev, delta);
}

extern "C" int b200dm_q_sample(const float* z, const float* sqrt_alpha_bar, const float* sqrt_one_minus_alpha_bar,
                               const int32_t* t, const float* noise, int64_t n_per_sample, int32_t batch, uint64_t seed,
                               int64_t sample_id0, void* x_t16, float* x_t32, void* stream) {
  B2_CHECK_ARG(z && sqrt_alpha_bar && sqrt_one_minus_alpha_bar && t && x_t16, "q_sample: null argument");
  B2_CHECK_ARG(n_per_sample > 0 && n_per_sample % 4 == 0 && batch > 0 && batch <= 65535, "q_sample: bad shape");
  const int64_t want = ((n_per_sample >> 2) + 255) / 256;
  int64_t cap = ((int64_t)b2_num_sms() * 8 + batch - 1) / batch;
  if (cap < 1) cap = 1;
  B2_CHECK_CUDA(b2_launch(q_sample_kernel, dim3((unsigned)(want < cap ? want : cap), (unsigned)batch), dim3(256), 0, (cudaStream_t)stream,
                          z, sqrt_alpha_bar, sqrt_one_minus_alpha_bar, t, noise, n_per_sample, seed, sample_id0, (act_t*)x_t16, x_t32));
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}

extern "C" size_t b200dm_noise_loss_workspace(int32_t batch) { return batch > 0 ? (size_t)batch * kLossBlocks * sizeof(double) : 0; }

extern "C" int b200dm_noise_loss(const float* eps_hat, const float* noise, int64_t n_per_sample, int32_t batch, int32_t channels,
                                 double divisor, uint64_t seed, int64_t sample_id0, float* loss, void* workspace, size_t ws_bytes,
                                 void* stream) {
  B2_CHECK_ARG(eps_hat && loss && workspace, "noise_loss: null argument");
  B2_CHECK_ARG(n_per_sample > 0 && n_per_sample % 4 == 0 && batch > 0 && batch <= 65535 && channels > 0 && divisor > 0.0,
               "noise_loss: bad arguments");
  B2_CHECK_ARG(ws_bytes >= b200dm_noise_loss_workspace(batch), "noise_loss: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;
  B2_CHECK_CUDA(b2_launch(sq_err_partial_kernel, dim3(kLossBlocks, (unsigned)batch), dim3(256), 0, s, eps_hat, noise, n_per_sample, seed,
                          sample_id0, (double*)workspace));
  // Keras MSE: mean over the channel axis, then the SUM reduction over (B, D, H, W); then / divisor
  B2_CHECK_CUDA(b2_launch(sq_err_final_kernel, dim3(1), dim3(1), 0, s, (const double*)workspace, (int)(batch * kLossBlocks),
                          1.0 / ((double)channels * divisor), loss));
  B2_CHECK_LAUNCH();
  return B200DM_OK;
}
