// Step program: an ordered list of kernel invocations over fixed buffers, replayed natively with one
// call per U-Net forward / decode (the reference drives one eager TF op at a time from Python,
// networks/dm3d.py:516-530).  Every launch goes to the caller's stream, so the whole program is
// CUDA-graph capturable; timestep-dependent inputs are read through device pointers (t_dev).
//
// Lanes: independent branches of a block (the three branches of CrossAttentionBlock.call all read the same tensor,
// conditional_dm3d.py:190-192) are recorded on side lanes = extra streams owned by the program, forked from / joined
// to the caller's stream with events (b200dm_program_add_sync), so under graph capture they become parallel branches
// and small kernels that fill a fraction of the 148 SMs overlap instead of queueing.
#include <memory>
#include <new>
#include "common.cuh"

namespace {
constexpr int kMaxLanes = 10;
struct Op {
  int lane = 0;                 // 0 = the caller's stream
  int to_lane = 0;              // sync op: lane that waits for everything recorded so far on `lane`
  cudaEvent_t ev = nullptr;     // set on sync ops only, which have no launches
  BoundOp bound;
};
}  // namespace

struct b200dm_program {
  std::vector<Op> ops;
  int cur_lane = 0;
  cudaStream_t side[kMaxLanes] = {};   // [0] unused
};

// add_X: bind op X exactly as b200dm_X would (same checks, codes and messages) and record it on the current lane; nothing is
// recorded on error.
template <typename Bind, typename... Args>
static int record(b200dm_program* p, const char* who, Bind bind, Args... args) {
  B2_CHECK_ARG(p, "%s: null program", who);
  Op op;
  op.lane = p->cur_lane;
  const int rc = bind(args..., &op.bound);
  if (rc == B200DM_OK) p->ops.push_back(std::move(op));
  return rc;
}

// Conv and attention plans are checked when they are created: the op is one launch of the plan, and owns it.
template <typename Plan>
static int bind_plan(Plan* plan, int (*run)(Plan*, void*), void (*destroy)(Plan*), BoundOp* op) {
  std::shared_ptr<Plan> owned(plan, destroy);
  op->launches.push_back([owned, run](cudaStream_t s) { return run(owned.get(), s); });
  return B200DM_OK;
}

extern "C" int b200dm_program_create(b200dm_program** out) {
  B2_CHECK_ARG(out, "program_create: null out");
  *out = new (std::nothrow) b200dm_program();
  B2_CHECK_ARG(*out, "program_create: out of memory");
  return B200DM_OK;
}

extern "C" void b200dm_program_destroy(b200dm_program* p) {
  if (!p) return;
  for (auto& op : p->ops)
    if (op.ev) cudaEventDestroy(op.ev);
  for (int i = 1; i < kMaxLanes; ++i)
    if (p->side[i]) cudaStreamDestroy(p->side[i]);
  delete p;
}

extern "C" int b200dm_program_add_conv(b200dm_program* p, b200dm_conv_plan* plan) {
  B2_CHECK_ARG(p && plan, "program_add_conv: null argument");
  return record(p, "program_add_conv", bind_plan<b200dm_conv_plan>, plan, b200dm_conv_plan_run, b200dm_conv_plan_destroy);
}

extern "C" int b200dm_program_add_attention(b200dm_program* p, b200dm_attn_plan* plan) {
  B2_CHECK_ARG(p && plan, "program_add_attention: null argument");
  return record(p, "program_add_attention", bind_plan<b200dm_attn_plan>, plan, b200dm_attention_plan_run, b200dm_attention_plan_destroy);
}

extern "C" int b200dm_program_add_norm_act_ex(b200dm_program* p, const b200dm_norm_ex_desc* d, const void* x, const float* a,
                                              const float* b, const float* mean_rstd, const void* prelu_alpha,
                                              const void* residual, void* y) {
  return record(p, "program_add_norm_act_ex", bind_norm_act_ex, d, x, a, b, mean_rstd, prelu_alpha, residual, y);
}

extern "C" int b200dm_program_add_stats_f32(b200dm_program* p, const float* x, int32_t batch, int64_t per_sample, float eps,
                                            float* mean_rstd, void* workspace, size_t ws_bytes) {
  return record(p, "program_add_stats_f32", bind_stats_f32, x, batch, per_sample, eps, mean_rstd, workspace, ws_bytes);
}

extern "C" int b200dm_program_add_norm_act(b200dm_program* p, const b200dm_norm_desc* d, const void* x0, const void* x1,
                                           const float* a, const float* b, const float* mean_rstd, void* y) {
  return record(p, "program_add_norm_act", bind_norm_act_fwd, d, x0, x1, a, b, mean_rstd, y);
}

extern "C" int b200dm_program_add_gn_stats(b200dm_program* p, const b200dm_norm_desc* d, const void* x, float eps,
                                           float* mean_rstd, float* workspace, size_t ws_bytes) {
  return record(p, "program_add_gn_stats", bind_gn_stats, d, x, eps, mean_rstd, workspace, ws_bytes);
}

extern "C" int b200dm_program_add_bn_stats(b200dm_program* p, const void* x, int64_t rows, int32_t c, const float* gamma,
                                           const float* beta, float eps, float* scale, float* shift, float* workspace, size_t ws_bytes) {
  return record(p, "program_add_bn_stats", bind_bn_stats, x, rows, c, gamma, beta, eps, scale, shift, workspace, ws_bytes);
}

extern "C" int b200dm_program_add_gn_finalize(b200dm_program* p, const double* partials, int32_t batch, int32_t rows_per_sample,
                                              int32_t c, int32_t groups, int64_t voxels_per_sample, float eps, float* mean_rstd) {
  return record(p, "program_add_gn_finalize", bind_gn_finalize, partials, batch, rows_per_sample, c, groups, voxels_per_sample, eps,
                mean_rstd);
}

extern "C" int b200dm_program_add_layernorm(b200dm_program* p, const void* x, int64_t rows, int32_t c, float eps,
                                            int32_t n_out, const float* const* gammas, const float* const* betas,
                                            void* const* ys) {
  return record(p, "program_add_layernorm", bind_layernorm_fwd, x, rows, c, eps, n_out, gammas, betas, ys);
}

extern "C" int b200dm_program_add_softmax(b200dm_program* p, const float* s, void* p_bf16, int64_t rows, int32_t cols,
                                          float scale) {
  return record(p, "program_add_softmax", bind_softmax_rows, s, p_bf16, rows, cols, scale);
}

extern "C" int b200dm_program_add_update(b200dm_program* p, const b200dm_update_desc* d, const float* x_t, const void* eps,
                                         const float* noise, float* x_prev, void* x_prev_bf16) {
  return record(p, "program_add_update", bind_ddpm_update, d, x_t, eps, noise, x_prev, x_prev_bf16);
}

extern "C" int b200dm_program_add_step_advance(b200dm_program* p, int32_t* t_dev, int32_t delta) {
  return record(p, "program_add_step_advance", bind_step_advance, t_dev, delta);
}

extern "C" int b200dm_program_set_lane(b200dm_program* p, int32_t lane) {
  B2_CHECK_ARG(p && lane >= 0 && lane < kMaxLanes, "program_set_lane: lane must be 0..%d", kMaxLanes - 1);
  if (lane > 0 && !p->side[lane]) B2_CHECK_CUDA(cudaStreamCreateWithFlags(&p->side[lane], cudaStreamNonBlocking));
  p->cur_lane = lane;
  return B200DM_OK;
}

extern "C" int b200dm_program_add_sync(b200dm_program* p, int32_t from_lane, int32_t to_lane) {
  B2_CHECK_ARG(p && from_lane >= 0 && from_lane < kMaxLanes && to_lane >= 0 && to_lane < kMaxLanes && from_lane != to_lane,
               "program_add_sync: bad lanes %d -> %d", from_lane, to_lane);
  for (int l : {from_lane, to_lane})
    if (l > 0 && !p->side[l]) B2_CHECK_CUDA(cudaStreamCreateWithFlags(&p->side[l], cudaStreamNonBlocking));
  Op op;
  B2_CHECK_CUDA(cudaEventCreateWithFlags(&op.ev, cudaEventDisableTiming));
  op.lane = from_lane; op.to_lane = to_lane;
  p->ops.push_back(std::move(op));
  return B200DM_OK;
}

extern "C" int b200dm_program_num_launches(const b200dm_program* p) {
  if (!p) return 0;
  int n = 0;
  for (const auto& op : p->ops) n += (int)op.bound.launches.size();
  return n;
}

static inline cudaStream_t lane_stream(b200dm_program* p, int lane, void* main) { return lane == 0 ? (cudaStream_t)main : p->side[lane]; }

extern "C" int b200dm_program_run(b200dm_program* p, void* stream) {
  B2_CHECK_ARG(p, "program_run: null program");
  for (auto& op : p->ops) {
    const cudaStream_t s = lane_stream(p, op.lane, stream);
    if (op.ev) {
      B2_CHECK_CUDA(cudaEventRecord(op.ev, s));
      B2_CHECK_CUDA(cudaStreamWaitEvent(lane_stream(p, op.to_lane, stream), op.ev, 0));
    } else if (const int rc = op.bound.run(s)) {
      return rc;
    }
  }
  return B200DM_OK;
}

// Same launches, with a CUDA event pair around every op on the launching stream; ms_per_op[i] = device time of
// op i.  Synchronises the stream (profiling aid for bench.py's roofline figures; not capturable).
extern "C" int b200dm_program_run_timed(b200dm_program* p, void* stream, float* ms_per_op, int32_t n_ops) {
  B2_CHECK_ARG(p && ms_per_op, "program_run_timed: null argument");
  B2_CHECK_ARG(n_ops == (int32_t)p->ops.size(), "program_run_timed: n_ops %d != %d", n_ops, (int)p->ops.size());
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<cudaEvent_t> ev(p->ops.size() + 1);
  for (auto& e : ev) B2_CHECK_CUDA(cudaEventCreate(&e));
  B2_CHECK_CUDA(cudaEventRecord(ev[0], s));
  int rc = B200DM_OK;
  for (size_t i = 0; i < p->ops.size() && rc == B200DM_OK; ++i) {   // every lane's ops serially on the caller's stream
    rc = p->ops[i].bound.run(s);
    cudaEventRecord(ev[i + 1], s);
  }
  cudaError_t e = cudaStreamSynchronize(s);
  if (rc == B200DM_OK && e == cudaSuccess)
    for (size_t i = 0; i < p->ops.size(); ++i) cudaEventElapsedTime(&ms_per_op[i], ev[i], ev[i + 1]);
  for (auto& x : ev) cudaEventDestroy(x);
  if (rc != B200DM_OK) return rc;
  B2_CHECK_CUDA(e);
  return B200DM_OK;
}

extern "C" int b200dm_program_num_ops(const b200dm_program* p) { return p ? (int)p->ops.size() : 0; }
