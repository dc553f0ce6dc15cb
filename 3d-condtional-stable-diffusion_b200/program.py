"""Python handle on a native step program (csrc/program.cu): an ordered list of kernel invocations over
fixed buffers.  Building happens once; ``run()`` is one ctypes call and is CUDA-graph capturable."""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib as L
from . import ops
from ._lib import lib, check, ptr, stream


class Program:
    def __init__(self, device):
        L.require_gpu()
        self.device = device
        h = C.c_void_p()
        check(lib().b200dm_program_create(C.byref(h)))
        self.h = h
        self.keep = []       # every tensor the program points at
        self.flops = 0.0     # algorithmic tensor-core FLOPs per run
        self.bytes = 0.0     # algorithmic HBM bytes of the elementwise ops per run
        self.log = []        # (kind, note) per op, for profiles / debugging
        self.outputs = {}    # note -> output tensor (layer-by-layer parity debugging)
        self.producers = {}  # data_ptr of a conv output -> its ConvPlan (gn_stats asks it for GroupNorm partial sums)
        self.op_bytes = {}   # note -> algorithmic HBM bytes of that conv launch

    # -- allocation helper
    def buf(self, shape, dtype=torch.bfloat16):
        t = torch.empty(tuple(shape), dtype=L.storage(dtype), device=self.device)
        self.keep.append(t)
        return t

    def hold(self, *ts):
        for t in ts:
            if t is not None:
                self.keep.append(t)
        return ts[0] if len(ts) == 1 else ts

    # -- ops
    def conv(self, desc, x0, w_packed, y, x1=None, bias=None, chan_bias=None, t_dev=None, residual=None,
             prelu_alpha=None, out_affine=None, shortcut=None, note=""):
        """``shortcut``: (x0, x1, w_packed, bias) of ConvPlan.set_shortcut; returns None, adding nothing, when the plan's
        kernel cannot carry it."""
        plan = ops.ConvPlan(desc, x0, w_packed, y, x1=x1, bias=bias, chan_bias=chan_bias, t_dev=t_dev,
                            residual=residual, prelu_alpha=prelu_alpha, out_affine=out_affine)
        if shortcut is not None and not plan.set_shortcut(*shortcut):
            return None
        check(lib().b200dm_program_add_conv(self.h, plan.h))
        plan.release()
        self.keep.extend(t for t in plan.keep if t is not None)
        kind = plan.info["halo"]
        self.op_bytes[note] = plan.alg_bytes
        if kind == 2:   # C_out = 1 stencil-reduce kernel: HBM-bound, accounted in bytes (input read once + output written)
            nbytes = float(x0.numel() * x0.element_size() + y.numel() * y.element_size())
            self.bytes += nbytes
            self.log.append(("stencil", note, nbytes))
        else:
            self.flops += plan.flops
            self.log.append(("conv_halo" if kind else "conv", note, plan.flops))
        self.outputs[note] = y
        self.producers[y.data_ptr()] = plan
        return y

    def norm_act(self, x0, a, b, y, act=None, x1=None, kind=0, groups=1, mean_rstd=None, note=""):
        d = ops.make_norm_desc(x0, x1, kind, groups, act)
        check(lib().b200dm_program_add_norm_act(self.h, C.byref(d), ptr(x0), ptr(x1), ptr(a), ptr(b), ptr(mean_rstd), ptr(y)))
        self.hold(x0, x1, a, b, mean_rstd, y)
        nbytes = 2.0 * y.numel() * 2
        self.bytes += nbytes
        self.log.append(("norm_act", note, nbytes))
        self.outputs[note] = y
        return y

    def gn_stats(self, x, groups, eps, note=""):
        """(mean, rstd) per (sample, group) of x -> fp32 (B, groups, 2).  When x is the output of a conv whose kernel can
        accumulate the sums in its epilogue (d-sweeping 32 -> 32 kernel), only a tiny fixed-order reduction is recorded;
        otherwise a statistics pass re-reads x."""
        plan = self.producers.get(x.data_ptr())
        part = plan.gn_partials() if plan is not None and x.dtype == L.ACT_DTYPE else None
        if part is not None:
            ws, rows = part
            mr = self.buf((x.shape[0], groups, 2), torch.float32)
            vox = x[0].numel() // x.shape[-1]
            check(lib().b200dm_program_add_gn_finalize(self.h, ptr(ws), x.shape[0], rows, x.shape[-1], groups, vox, eps, ptr(mr)))
            self.hold(ws, x)
            self.log.append(("gn_stats", note + " (from the conv epilogue)", 0.0))
            return mr
        d = ops.make_norm_desc(x, None, 1, groups)
        ws_bytes = lib().b200dm_gn_stats_workspace(C.byref(d))
        ws = self.buf((ws_bytes // 4,), torch.float32)
        mr = self.buf((x.shape[0], groups, 2), torch.float32)
        check(lib().b200dm_program_add_gn_stats(self.h, C.byref(d), ptr(x), eps, ptr(mr), ptr(ws), ws_bytes))
        self.hold(x)
        self.bytes += x.numel() * 2.0
        self.log.append(("gn_stats", note, x.numel() * 2.0))
        return mr

    def bn_stats(self, x, gamma, beta, scale, shift, eps=1e-3, note=""):
        """scale / shift (fp32 (C,) views) <- BatchNorm coefficients from the batch statistics of x (training=True); two reads
        of x."""
        c = x.shape[-1]
        ws_bytes = lib().b200dm_bn_stats_workspace(c)
        ws = self.buf((ws_bytes // 4,), torch.float32)
        check(lib().b200dm_program_add_bn_stats(self.h, ptr(x), x.numel() // c, c, ptr(gamma), ptr(beta), eps, ptr(scale), ptr(shift),
                                                ptr(ws), ws_bytes))
        self.hold(x, gamma, beta, scale, shift)
        self.bytes += x.numel() * 4.0
        self.log.append(("bn_stats", note, x.numel() * 4.0))
        return scale, shift

    def norm_act_ex(self, x, a, b, y, kind=0, groups=1, mean_rstd=None, prelu_alpha=None, residual=None, act=None, post_act=None,
                    upsample=False, note=""):
        """y = post_act(residual + act(PReLU(norm(x)))), x optionally nearest-upsampled x2; y (B,D,H,W,C) bf16 | fp32."""
        d = L.NormExDesc()
        d.batch, d.out_d, d.out_h, d.out_w, d.c = y.shape
        d.kind, d.groups, d.act, d.post_act, d.upsample = kind, groups, L.ACT[act], L.ACT[post_act], int(upsample)
        d.x_dtype, d.y_dtype = L.dt(x), L.dt(y)
        check(lib().b200dm_program_add_norm_act_ex(self.h, C.byref(d), ptr(x), ptr(a), ptr(b), ptr(mean_rstd), ptr(prelu_alpha),
                                                   ptr(residual), ptr(y)))
        self.hold(x, a, b, mean_rstd, prelu_alpha, residual, y)
        nbytes = float(x.numel() * x.element_size() + y.numel() * y.element_size() +
                       (prelu_alpha.numel() * 2 if prelu_alpha is not None else 0) + (residual.numel() * 2 if residual is not None else 0))
        self.bytes += nbytes
        self.log.append(("norm_act", note, nbytes))
        self.outputs[note] = y
        return y

    def stats_f32(self, x, eps, note=""):
        """(mean, rstd) over each whole sample of an fp32 tensor -> fp32 (B, 1, 2)."""
        B = x.shape[0]
        ws_bytes = lib().b200dm_stats_f32_workspace(B)
        ws = self.buf((ws_bytes // 8,), torch.float64)
        mr = self.buf((B, 1, 2), torch.float32)
        check(lib().b200dm_program_add_stats_f32(self.h, ptr(x), B, x[0].numel(), eps, ptr(mr), ptr(ws), ws_bytes))
        self.hold(x)
        self.bytes += x.numel() * 4.0
        self.log.append(("gn_stats", note, x.numel() * 4.0))
        return mr

    def layernorm(self, x, gammas, betas, ys, eps=1e-3, note=""):
        c = x.shape[-1]
        check(lib().b200dm_program_add_layernorm(self.h, ptr(x), x.numel() // c, c, eps, len(gammas), ops._ptr_array(gammas),
                                                 ops._ptr_array(betas), ops._ptr_array(ys)))
        self.hold(x, *gammas, *betas, *ys)
        self.bytes += x.numel() * 2.0 * (1 + len(ys))
        self.log.append(("layernorm", note, x.numel() * 2.0 * (1 + len(ys))))
        return ys

    def attention(self, q, k, vt, o, scale, residual=None, note=""):
        plan = ops.AttnPlan(q, k, vt, o, scale, residual)
        self.flops += plan.flops
        check(lib().b200dm_program_add_attention(self.h, plan.h))
        plan.release()
        self.hold(q, k, vt, o, residual)
        self.log.append(("attn", note, plan.flops))
        self.outputs[note] = o
        return o

    def softmax(self, s, p, scale, note=""):
        cols = s.shape[-1]
        check(lib().b200dm_program_add_softmax(self.h, ptr(s), ptr(p), s.numel() // cols, cols, scale))
        self.hold(s, p)
        self.bytes += s.numel() * 6.0
        self.log.append(("softmax", note, s.numel() * 6.0))
        return p

    def update(self, desc, x_t, eps, x_prev, x_prev_bf16=None, noise=None, note=""):
        check(lib().b200dm_program_add_update(self.h, C.byref(desc), ptr(x_t), ptr(eps), ptr(noise), ptr(x_prev), ptr(x_prev_bf16)))
        self.hold(x_t, eps, x_prev, x_prev_bf16, noise)
        nbytes = x_t.numel() * (4.0 + eps.element_size() + 4.0 + (2.0 if x_prev_bf16 is not None else 0.0))
        self.bytes += nbytes
        self.log.append(("update", note, nbytes))

    def set_lane(self, lane):
        """Ops added from here on run on lane ``lane`` (0 = caller's stream; 1..3 = side streams of the program)."""
        check(lib().b200dm_program_set_lane(self.h, lane))

    def sync(self, from_lane, to_lane):
        """Everything recorded so far on ``from_lane`` becomes a prerequisite of what follows on ``to_lane``."""
        check(lib().b200dm_program_add_sync(self.h, from_lane, to_lane))
        self.log.append(("sync", f"{from_lane}->{to_lane}", 0))

    def advance(self, t_dev, delta):
        check(lib().b200dm_program_add_step_advance(self.h, ptr(t_dev), delta))
        self.hold(t_dev)
        self.log.append(("advance", "", 0))

    @property
    def num_launches(self):
        return lib().b200dm_program_num_launches(self.h)

    def run(self):
        check(lib().b200dm_program_run(self.h, stream()))

    def run_timed(self):
        """-> [(kind, note, work, ms)] per op (CUDA events around every launch; synchronises)."""
        n = lib().b200dm_program_num_ops(self.h)
        ms = (C.c_float * n)()
        check(lib().b200dm_program_run_timed(self.h, stream(), ms, n))
        assert n == len(self.log)
        return [(k, note, work, ms[i]) for i, (k, note, work) in enumerate(self.log)]

    def __del__(self):
        try:
            if getattr(self, "h", None):
                lib().b200dm_program_destroy(self.h)
                self.h = None
        except Exception:  # interpreter shutdown
            pass
