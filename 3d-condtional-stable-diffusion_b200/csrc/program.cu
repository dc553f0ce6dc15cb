// Step program: an ordered list of kernel invocations over fixed buffers, replayed natively with one
// call per U-Net forward / decode (the reference drives one eager TF op at a time from Python,
// networks/dm3d.py:516-530).  Every launch goes to the caller's stream, so the whole program is
// CUDA-graph capturable; timestep-dependent inputs are read through device pointers (t_dev).
//
// Lanes: independent branches of a block (the three branches of CrossAttentionBlock.call all read the same tensor,
// conditional_dm3d.py:190-192) are recorded on side lanes = extra streams owned by the program, forked from / joined
// to the caller's stream with events (b200dm_program_add_sync), so under graph capture they become parallel branches
// and small kernels that fill a fraction of the 148 SMs overlap instead of queueing.
#include <vector>
#include <new>
#include "common.cuh"

namespace {
enum OpKind { OP_CONV, OP_NORM, OP_GNSTATS, OP_LN, OP_SOFTMAX, OP_UPDATE, OP_ADVANCE, OP_ATTN, OP_NORM_EX, OP_STATS_F32, OP_SYNC, OP_GN_FINAL, OP_BN_STATS };
constexpr int kMaxLanes = 10;
struct Op {
  OpKind kind;
  int lane = 0;                 // 0 = the caller's stream
  int to_lane = 0;              // OP_SYNC: lane that waits for everything recorded so far on `lane`
  cudaEvent_t ev = nullptr;     // OP_SYNC
  b200dm_conv_plan* conv = nullptr;
  b200dm_attn_plan* attn = nullptr;
  b200dm_norm_desc nd{};
  b200dm_norm_ex_desc ned{};
  const void* p5 = nullptr;
  b200dm_update_desc ud{};
  const void* p0 = nullptr; const void* p1 = nullptr; const void* p2 = nullptr; const void* p3 = nullptr; const void* p4 = nullptr;
  void* out = nullptr; void* out2 = nullptr;
  float f0 = 0.f;
  int64_t i0 = 0; int32_t i1 = 0, i2 = 0;
  size_t ws = 0;
  const float* gam[3] = {nullptr, nullptr, nullptr};
  const float* bet[3] = {nullptr, nullptr, nullptr};
  void* ys[3] = {nullptr, nullptr, nullptr};
  int launches = 1;
};
}  // namespace

struct b200dm_program {
  std::vector<Op> ops;
  int cur_lane = 0;
  cudaStream_t side[kMaxLanes] = {};   // [0] unused
  void push(Op& op) { op.lane = cur_lane; ops.push_back(op); }
};

extern "C" int b200dm_program_create(b200dm_program** out) {
  B2_CHECK_ARG(out, "program_create: null out");
  *out = new (std::nothrow) b200dm_program();
  B2_CHECK_ARG(*out, "program_create: out of memory");
  return B200DM_OK;
}

extern "C" void b200dm_program_destroy(b200dm_program* p) {
  if (!p) return;
  for (auto& op : p->ops)
    if (op.kind == OP_CONV) b200dm_conv_plan_destroy(op.conv);
    else if (op.kind == OP_ATTN) b200dm_attention_plan_destroy(op.attn);
    else if (op.kind == OP_SYNC && op.ev) cudaEventDestroy(op.ev);
  for (int i = 1; i < kMaxLanes; ++i)
    if (p->side[i]) cudaStreamDestroy(p->side[i]);
  delete p;
}

extern "C" int b200dm_program_add_conv(b200dm_program* p, b200dm_conv_plan* plan) {
  B2_CHECK_ARG(p && plan, "program_add_conv: null argument");
  Op op; op.kind = OP_CONV; op.conv = plan;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_norm_act_ex(b200dm_program* p, const b200dm_norm_ex_desc* d, const void* x, const float* a,
                                              const float* b, const float* mean_rstd, const void* prelu_alpha,
                                              const void* residual, void* y) {
  B2_CHECK_ARG(p && d && x && a && b && y, "program_add_norm_act_ex: null argument");
  Op op; op.kind = OP_NORM_EX; op.ned = *d; op.p0 = x; op.p1 = a; op.p2 = b; op.p3 = mean_rstd; op.p4 = prelu_alpha; op.p5 = residual;
  op.out = y;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_stats_f32(b200dm_program* p, const float* x, int32_t batch, int64_t per_sample, float eps,
                                            float* mean_rstd, void* workspace, size_t ws_bytes) {
  B2_CHECK_ARG(p && x && mean_rstd && workspace, "program_add_stats_f32: null argument");
  Op op; op.kind = OP_STATS_F32; op.p0 = x; op.i1 = batch; op.i0 = per_sample; op.f0 = eps; op.out = mean_rstd; op.out2 = workspace;
  op.ws = ws_bytes; op.launches = 2;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_attention(b200dm_program* p, b200dm_attn_plan* plan) {
  B2_CHECK_ARG(p && plan, "program_add_attention: null argument");
  Op op; op.kind = OP_ATTN; op.attn = plan;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_norm_act(b200dm_program* p, const b200dm_norm_desc* d, const void* x0, const void* x1,
                                           const float* a, const float* b, const float* mean_rstd, void* y) {
  B2_CHECK_ARG(p && d && x0 && a && b && y, "program_add_norm_act: null argument");
  Op op; op.kind = OP_NORM; op.nd = *d; op.p0 = x0; op.p1 = x1; op.p2 = a; op.p3 = b; op.p4 = mean_rstd; op.out = y;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_gn_stats(b200dm_program* p, const b200dm_norm_desc* d, const void* x, float eps,
                                           float* mean_rstd, float* workspace, size_t ws_bytes) {
  B2_CHECK_ARG(p && d && x && mean_rstd && workspace, "program_add_gn_stats: null argument");
  Op op; op.kind = OP_GNSTATS; op.nd = *d; op.p0 = x; op.f0 = eps; op.out = mean_rstd; op.out2 = workspace; op.ws = ws_bytes;
  op.launches = 2;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_bn_stats(b200dm_program* p, const void* x, int64_t rows, int32_t c, const float* gamma,
                                           const float* beta, float eps, float* scale, float* shift, float* workspace, size_t ws_bytes) {
  B2_CHECK_ARG(p && x && gamma && beta && scale && shift && workspace, "program_add_bn_stats: null argument");
  Op op; op.kind = OP_BN_STATS; op.p0 = x; op.i0 = rows; op.i1 = c; op.p1 = gamma; op.p2 = beta; op.f0 = eps; op.out = scale;
  op.out2 = shift; op.p3 = workspace; op.ws = ws_bytes; op.launches = 4;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_gn_finalize(b200dm_program* p, const float* partials, int32_t batch, int32_t rows_per_sample,
                                              int32_t c, int32_t groups, int64_t voxels_per_sample, float eps, float* mean_rstd) {
  B2_CHECK_ARG(p && partials && mean_rstd, "program_add_gn_finalize: null argument");
  Op op; op.kind = OP_GN_FINAL; op.p0 = partials; op.i1 = batch; op.i2 = rows_per_sample; op.nd.c0 = c; op.nd.groups = groups;
  op.i0 = voxels_per_sample; op.f0 = eps; op.out = mean_rstd;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_layernorm(b200dm_program* p, const void* x, int64_t rows, int32_t c, float eps,
                                            int32_t n_out, const float* const* gammas, const float* const* betas,
                                            void* const* ys) {
  B2_CHECK_ARG(p && x && gammas && betas && ys && n_out >= 1 && n_out <= 3, "program_add_layernorm: bad argument");
  Op op; op.kind = OP_LN; op.p0 = x; op.i0 = rows; op.i1 = c; op.f0 = eps; op.i2 = n_out;
  for (int i = 0; i < n_out; ++i) { op.gam[i] = gammas[i]; op.bet[i] = betas[i]; op.ys[i] = ys[i]; }
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_softmax(b200dm_program* p, const float* s, void* p_bf16, int64_t rows, int32_t cols,
                                          float scale) {
  B2_CHECK_ARG(p && s && p_bf16, "program_add_softmax: null argument");
  Op op; op.kind = OP_SOFTMAX; op.p0 = s; op.out = p_bf16; op.i0 = rows; op.i1 = cols; op.f0 = scale;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_update(b200dm_program* p, const b200dm_update_desc* d, const float* x_t, const void* eps,
                                         const float* noise, float* x_prev, void* x_prev_bf16) {
  B2_CHECK_ARG(p && d && x_t && eps && x_prev, "program_add_update: null argument");
  Op op; op.kind = OP_UPDATE; op.ud = *d; op.p0 = x_t; op.p1 = eps; op.p2 = noise; op.out = x_prev; op.out2 = x_prev_bf16;
  p->push(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_add_step_advance(b200dm_program* p, int32_t* t_dev, int32_t delta) {
  B2_CHECK_ARG(p && t_dev, "program_add_step_advance: null argument");
  Op op; op.kind = OP_ADVANCE; op.out = t_dev; op.i1 = delta;
  p->push(op);
  return B200DM_OK;
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
  Op op; op.kind = OP_SYNC; op.launches = 0;
  B2_CHECK_CUDA(cudaEventCreateWithFlags(&op.ev, cudaEventDisableTiming));
  op.lane = from_lane; op.to_lane = to_lane;
  p->ops.push_back(op);
  return B200DM_OK;
}

extern "C" int b200dm_program_num_launches(const b200dm_program* p) {
  if (!p) return 0;
  int n = 0;
  for (const auto& op : p->ops) n += op.launches;
  return n;
}

static int run_op(Op& op, void* stream);

static inline cudaStream_t lane_stream(b200dm_program* p, int lane, void* main) { return lane == 0 ? (cudaStream_t)main : p->side[lane]; }

static int run_any(b200dm_program* p, Op& op, void* stream) {
  if (op.kind == OP_SYNC) {
    B2_CHECK_CUDA(cudaEventRecord(op.ev, lane_stream(p, op.lane, stream)));
    B2_CHECK_CUDA(cudaStreamWaitEvent(lane_stream(p, op.to_lane, stream), op.ev, 0));
    return B200DM_OK;
  }
  return run_op(op, (void*)lane_stream(p, op.lane, stream));
}

extern "C" int b200dm_program_run(b200dm_program* p, void* stream) {
  B2_CHECK_ARG(p, "program_run: null program");
  for (auto& op : p->ops) {
    int rc = run_any(p, op, stream);
    if (rc != B200DM_OK) return rc;
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
    if (p->ops[i].kind != OP_SYNC) rc = run_op(p->ops[i], stream);
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

static int run_op(Op& op, void* stream) {
  int rc = B200DM_OK;
  {
    switch (op.kind) {
      case OP_CONV: rc = b200dm_conv_plan_run(op.conv, stream); break;
      case OP_NORM:
        rc = b200dm_norm_act_fwd(&op.nd, op.p0, op.p1, (const float*)op.p2, (const float*)op.p3, (const float*)op.p4, op.out, stream);
        break;
      case OP_GNSTATS: rc = b200dm_gn_stats(&op.nd, op.p0, op.f0, (float*)op.out, (float*)op.out2, op.ws, stream); break;
      case OP_LN: rc = b200dm_layernorm_fwd(op.p0, op.i0, op.i1, op.f0, op.i2, op.gam, op.bet, op.ys, stream); break;
      case OP_SOFTMAX: rc = b200dm_softmax_rows((const float*)op.p0, op.out, op.i0, op.i1, op.f0, stream); break;
      case OP_UPDATE:
        rc = b200dm_ddpm_update(&op.ud, (const float*)op.p0, op.p1, (const float*)op.p2, (float*)op.out, op.out2, stream);
        break;
      case OP_ADVANCE: rc = b200dm_step_advance((int32_t*)op.out, op.i1, stream); break;
      case OP_ATTN: rc = b200dm_attention_plan_run(op.attn, stream); break;
      case OP_NORM_EX:
        rc = b200dm_norm_act_ex(&op.ned, op.p0, (const float*)op.p1, (const float*)op.p2, (const float*)op.p3, op.p4, op.p5, op.out, stream);
        break;
      case OP_SYNC: break;
      case OP_GN_FINAL:
        rc = b200dm_gn_finalize((const float*)op.p0, op.i1, op.i2, op.nd.c0, op.nd.groups, op.i0, op.f0, (float*)op.out, stream);
        break;
      case OP_BN_STATS:
        rc = b200dm_bn_stats(op.p0, op.i0, op.i1, (const float*)op.p1, (const float*)op.p2, op.f0, (float*)op.out, (float*)op.out2,
                             (float*)op.p3, op.ws, stream);
        break;
      case OP_STATS_F32: rc = b200dm_stats_f32((const float*)op.p0, op.i1, op.i0, op.f0, (float*)op.out, op.out2, op.ws, stream); break;
    }
  }
  return rc;
}
