// Shared helpers for libb200dm (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <functional>
#include <vector>
#include "../../include/b200dm.h"

void b200dm_set_error(const char* fmt, ...);

// ---- 16-bit activation / weight storage type ------------------------------------------------------------
// The library is built twice from the same sources: libb200dm.so stores activations and packed weights as bf16
// (8 significand bits, fp32 range), libb200dm_f16.so (-DB200DM_ACT_FP16) as IEEE fp16 (11 significand bits: 8x smaller
// storage rounding, range 65504).  tcgen05.mma kind::f16 runs both at the same rate and always accumulates in fp32.
#ifdef B200DM_ACT_FP16
typedef __half act_t;
typedef __half2 act2_t;
__device__ __forceinline__ float2 act2_to_float2(const act2_t v) { return __half22float2(v); }
__device__ __forceinline__ act2_t floats_to_act2(float a, float b) { return __floats2half2_rn(a, b); }
__device__ __forceinline__ float act_to_float(const act_t v) { return __half2float(v); }
__device__ __forceinline__ act_t float_to_act(float v) { return __float2half_rn(v); }
#define B200DM_ACT_NAME "fp16"
#else
typedef __nv_bfloat16 act_t;
typedef __nv_bfloat162 act2_t;
__device__ __forceinline__ float2 act2_to_float2(const act2_t v) { return __bfloat1622float2(v); }
__device__ __forceinline__ act2_t floats_to_act2(float a, float b) { return __floats2bfloat162_rn(a, b); }
__device__ __forceinline__ float act_to_float(const act_t v) { return __bfloat162float(v); }
__device__ __forceinline__ act_t float_to_act(float v) { return __float2bfloat16_rn(v); }
#define B200DM_ACT_NAME "bf16"
#endif

#define B2_CHECK_ARG(cond, ...)                 \
  do {                                          \
    if (!(cond)) {                              \
      b200dm_set_error(__VA_ARGS__);            \
      return B200DM_ERR_INVALID;                \
    }                                           \
  } while (0)

#define B2_CHECK_CUDA(expr)                                                                  \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      b200dm_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return B200DM_ERR_CUDA;                                                                \
    }                                                                                        \
  } while (0)

#define B2_CHECK_LAUNCH() B2_CHECK_CUDA(cudaGetLastError())

static inline int b2_num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

// ---- programmatic dependent launch (PDL) ----------------------------------------------------------------
// Every per-step kernel calls pdl_launch_dependents() first (the next kernel of the stream / graph may start its
// prologue as soon as all CTAs of this one are resident) and pdl_wait() before its first access to global memory that
// a predecessor may have written (or may still read): barrier init, TMEM allocation, tensor-map prefetch and launch
// latency of kernel k+1 overlap the tail of kernel k.  B200DM_PDL=0 launches without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

bool b200dm_pdl_enabled();

// cluster: CTAs per thread-block cluster along x (1 = no cluster)
template <typename... KArgs, typename... Args>
static inline cudaError_t b2_launch_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, unsigned cluster, size_t smem, cudaStream_t s,
                                            Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[2];
  unsigned n = 0;
  if (cluster > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = cluster; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
    ++n;
  }
  if (b200dm_pdl_enabled()) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = at; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

template <typename... KArgs, typename... Args>
static inline cudaError_t b2_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  return b2_launch_cluster(kern, grid, block, 1u, smem, s, args...);
}

// ---- bound ops ------------------------------------------------------------------------------------------------------
// An op ready to launch: kernel launches with grid, block, dynamic shared memory and arguments fixed.  bind_X(args..., op)
// does all of b200dm_X(args..., stream) that comes before its first launch -- argument checks (same codes and messages), grid
// and shared-memory sizing -- without a stream; b200dm_X is bind_X + run(), and a step program records and replays the op.
struct BoundOp {
  std::vector<std::function<int(cudaStream_t)>> launches;   // each returns a B200DM_* code
  int run(cudaStream_t s) const {
    for (const auto& launch : launches)
      if (const int rc = launch(s)) return rc;
    B2_CHECK_LAUNCH();
    return B200DM_OK;
  }
};

// static: the closure may capture a kernel argument type of a .cu file's anonymous namespace
template <typename... KArgs, typename... Args>
static void bind_launch(BoundOp* op, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args) {
  op->launches.push_back([=](cudaStream_t s) -> int {
    B2_CHECK_CUDA(b2_launch(kern, grid, block, smem, s, args...));
    return B200DM_OK;
  });
}

template <typename Bind, typename... Args>
int bind_and_run(Bind bind, void* stream, Args... args) {
  BoundOp op;
  const int rc = bind(args..., &op);
  return rc ? rc : op.run((cudaStream_t)stream);
}

int bind_norm_act_fwd(const b200dm_norm_desc* d, const void* x0, const void* x1, const float* a, const float* b,
                      const float* mean_rstd, void* y, BoundOp* op);
int bind_gn_stats(const b200dm_norm_desc* d, const void* x, float eps, float* mean_rstd, float* workspace, size_t ws_bytes, BoundOp* op);
int bind_bn_stats(const void* x, int64_t rows, int32_t c, const float* gamma, const float* beta, float eps, float* scale,
                  float* shift, float* workspace, size_t ws_bytes, BoundOp* op);
int bind_gn_finalize(const double* partials, int32_t batch, int32_t rows_per_sample, int32_t c, int32_t groups,
                     int64_t voxels_per_sample, float eps, float* mean_rstd, BoundOp* op);
int bind_layernorm_fwd(const void* x, int64_t rows, int32_t c, float eps, int32_t n_out, const float* const* gammas,
                       const float* const* betas, void* const* ys, BoundOp* op);
int bind_norm_act_ex(const b200dm_norm_ex_desc* d, const void* x, const float* a, const float* b, const float* mean_rstd,
                     const void* prelu_alpha, const void* residual, void* y, BoundOp* op);
int bind_stats_f32(const float* x, int32_t batch, int64_t per_sample, float eps, float* mean_rstd, void* workspace, size_t ws_bytes, BoundOp* op);
int bind_softmax_rows(const float* s, void* p_bf16, int64_t rows, int32_t cols, float scale, BoundOp* op);
int bind_ddpm_update(const b200dm_update_desc* d, const float* x_t, const void* eps, const float* noise, float* x_prev,
                     void* x_prev_bf16, BoundOp* op);
int bind_step_advance(int32_t* t_dev, int32_t delta, BoundOp* op);

// ---- TMA descriptors ----------------------------------------------------------------------------------------------
// Opt-in limit of one block's dynamic shared memory on sm_100 (227 KB).
constexpr size_t kMaxDynamicSmem = 232448;

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda); nullptr without a driver.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn b2_encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  }
  return fn;
}

// ---- small device helpers ------------------------------------------------------------------
struct __align__(16) bf16x8 {
  act2_t v[4];
};

__device__ __forceinline__ bf16x8 ldg_bf16x8(const bf16x8* p) {   // 16-byte read-only load
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  bf16x8 r;
  memcpy(&r, &u, 16);
  return r;
}
__device__ __forceinline__ void unpack8(const bf16x8& p, float (&f)[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = act2_to_float2(p.v[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ bf16x8 pack8(const float (&f)[8]) {
  bf16x8 p;
#pragma unroll
  for (int i = 0; i < 4; ++i) p.v[i] = floats_to_act2(f[2 * i], f[2 * i + 1]);
  return p;
}
// x * sigmoid(x).  ex2.approx.ftz == __expf outside the denormal range, and there 1 + e == 1 either way: same values as
// __fdividef(x, 1 + __expf(-x)) without the per-element range fix-up (FSETP + two predicated FMULs) of the non-ftz form.
__device__ __forceinline__ float silu_f(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
  return __fdividef(x, 1.0f + e);
}
__device__ __forceinline__ float apply_act(float x, int act) {
  if (act == B200DM_ACT_SILU) return silu_f(x);
  if (act == B200DM_ACT_RELU) return fmaxf(x, 0.0f);
  return x;
}
// Runtime activation of a register vector with the kind test OUTSIDE the element loop.  With the test inside, the compiler
// emitted a branch per element and the N dependent MUFU.EX2 -> FADD -> MUFU.RCP -> FMUL chains ran one after the other
// (~80 cycles each): the SiLU epilogue of a 64 -> 64 conv tile took 9.3 k cycles against 3.6 k without activation and made
// the ResidualBlock conv1 launches epilogue-bound (clock64 timeline, tools/conv_trace.py EPI=1).
template <int N>
__device__ __forceinline__ void apply_act_vec(float (&v)[N], int act) {
  if (act == B200DM_ACT_SILU) {
#pragma unroll
    for (int j = 0; j < N; ++j) v[j] = silu_f(v[j]);
  } else if (act == B200DM_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < N; ++j) v[j] = fmaxf(v[j], 0.0f);
  }
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
