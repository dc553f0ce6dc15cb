"""Tensor-level wrappers over the C ABI (one function per entry point of include/b200dm.h).

Layout: activations are channels-last (N, D, H, W, C) like the reference's; bf16 on the hot path,
fp32 for x_t / eps_hat / decoded volumes.  All functions enqueue on torch's current stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L
from ._lib import lib, check, ptr, stream, dt


def _dev():
    L.require_gpu()
    return torch.device("cuda", torch.cuda.current_device())


# ------------------------------------------------------------------ K10 update
class ScheduleTables:
    """Device copies of the reference's ``Betas`` tables (networks/dm3d.py:194-214): float64 numpy -> float32."""

    NAMES = ("beta", "sqrt_alpha", "alpha_bar", "alpha_bar_prev", "sqrt_alpha_bar", "sqrt_alpha_bar_prev",
             "sqrt_one_minus_alpha_bar")

    def __init__(self, timesteps: int, device=None):
        beta = np.linspace(0.0001, 0.02, timesteps)
        alpha = 1 - beta
        alpha_bar = np.cumprod(alpha, 0)
        alpha_bar_prev = np.append(1.0, alpha_bar[:-1])
        host = dict(beta=beta, alpha=alpha, sqrt_alpha=np.sqrt(alpha), alpha_bar=alpha_bar,
                    alpha_bar_prev=alpha_bar_prev, sqrt_alpha_bar=np.sqrt(alpha_bar),
                    sqrt_alpha_bar_prev=np.sqrt(alpha_bar_prev), sqrt_one_minus_alpha_bar=np.sqrt(1 - alpha_bar))
        self.timesteps = timesteps
        self.host = {k: np.asarray(v, dtype=np.float32) for k, v in host.items()}
        self.dev = None
        if device is not None:
            self.to(device)

    def to(self, device):
        self.dev = {k: torch.from_numpy(v).to(device) for k, v in self.host.items()}
        return self

    def fill(self, d: L.UpdateDesc):
        for n in self.NAMES:
            setattr(d, n, self.dev[n].data_ptr())


def make_update_desc(tables: ScheduleTables, n_per_sample, batch, t=0, t_prev=-1, sampler=0, seed=0, sample_id0=0,
                     eps_dtype=L.F32, t_dev=None, seed_on_device=False) -> L.UpdateDesc:
    d = L.UpdateDesc()
    d.n_per_sample, d.batch, d.sampler = n_per_sample, batch, sampler
    tables.fill(d)
    d.t_dev = t_dev.data_ptr() if t_dev is not None else None
    d.t, d.t_prev, d.seed, d.sample_id0, d.eps_dtype = t, t_prev, seed, sample_id0, eps_dtype
    d.reserved = 1 if seed_on_device else 0   # Philox key / sample base read from t_dev[4..7] (int32[8])
    return d


def ddpm_update(tables, x_t, eps, t, noise=None, seed=0, sample_id0=0, sampler=0, t_prev=-1, want_bf16=False):
    """One reverse step: DiffusionModel.sample + clip + noise add (dm3d.py:477-508, 528-530)."""
    _dev()
    assert x_t.dtype == torch.float32 and x_t.is_contiguous() and eps.is_contiguous()
    B = x_t.shape[0]
    n = x_t[0].numel()
    d = make_update_desc(tables, n, B, t, t_prev, sampler, seed, sample_id0, dt(eps))
    out = torch.empty_like(x_t)
    out_b = torch.empty(x_t.shape, dtype=L.ACT_DTYPE, device=x_t.device) if want_bf16 else None
    check(lib().b200dm_ddpm_update(C.byref(d), ptr(x_t), ptr(eps), ptr(noise), ptr(out), ptr(out_b), stream()))
    return (out, out_b) if want_bf16 else out


def q_sample(tables, z, t_dev, noise=None, seed=0, sample_id0=0, want_f32=False, out16=None):
    """x_t = sqrt(abar_t) z + sqrt(1 - abar_t) noise (train_step, conditional_dm3d.py:481-490) for per-sample ``t_dev`` (B,) int32
    on the device; the noise is Philox stream 2 of ``seed`` unless injected.  -> 16-bit x_t (and fp32 x_t when ``want_f32``)."""
    L.check_storage(z, noise, out16)
    _dev()
    assert z.dtype == torch.float32 and z.is_contiguous() and t_dev.dtype == torch.int32
    if out16 is None:
        out16 = torch.empty(z.shape, dtype=L.ACT_DTYPE, device=z.device)
    x32 = torch.empty_like(z) if want_f32 else None
    check(lib().b200dm_q_sample(ptr(z), ptr(tables.dev["sqrt_alpha_bar"]), ptr(tables.dev["sqrt_one_minus_alpha_bar"]), ptr(t_dev),
                                ptr(noise), z[0].numel(), z.shape[0], seed, sample_id0, ptr(out16), ptr(x32), stream()))
    return (out16, x32) if want_f32 else out16


def noise_loss(eps_hat, divisor, noise=None, seed=0, sample_id0=0):
    """MSE(reduction=SUM)(noise, eps_hat) / divisor (conditional_dm3d.py:496-499): mean over the last axis, sum over the rest.
    The noise is regenerated from q_sample's stream unless injected.  -> fp32 (1,) on the device."""
    L.check_storage(eps_hat, noise)
    _dev()
    assert eps_hat.dtype == torch.float32 and eps_hat.is_contiguous()
    B = eps_hat.shape[0]
    ws = torch.empty(lib().b200dm_noise_loss_workspace(B) // 8, dtype=torch.float64, device=eps_hat.device)
    loss = torch.empty(1, dtype=torch.float32, device=eps_hat.device)
    check(lib().b200dm_noise_loss(ptr(eps_hat), ptr(noise), eps_hat[0].numel(), B, eps_hat.shape[-1], float(divisor), seed, sample_id0,
                                  ptr(loss), ptr(ws), ws.numel() * 8, stream()))
    return loss


def philox_normal(shape, seed, sample_id0=0, step=0, stream_id=1, want_bf16=False):
    dev = _dev()
    x = torch.empty(shape, dtype=torch.float32, device=dev)
    xb = torch.empty(shape, dtype=L.ACT_DTYPE, device=dev) if want_bf16 else None
    check(lib().b200dm_philox_normal(ptr(x), ptr(xb), x[0].numel(), shape[0], seed, sample_id0, step, stream_id, stream()))
    return (x, xb) if want_bf16 else x


# ------------------------------------------------------------------ K6/K7 norms
def bn_fold(gamma, beta, mean, var, eps=1e-3):
    _dev()
    scale, shift = torch.empty_like(gamma), torch.empty_like(gamma)
    check(lib().b200dm_bn_fold(ptr(gamma), ptr(beta), ptr(mean), ptr(var), eps, gamma.numel(), ptr(scale), ptr(shift), stream()))
    return scale, shift


def bn_stats(x, gamma, beta, eps=1e-3, scale=None, shift=None):
    """BatchNormalization with the batch's own statistics (training=True): x (..., C) 16-bit -> (scale, shift) fp32 (C,), the
    per-channel affine of norm_act / the conv epilogue."""
    L.check_storage(x)
    _dev()
    c = x.shape[-1]
    scale = torch.empty(c, dtype=torch.float32, device=x.device) if scale is None else scale
    shift = torch.empty(c, dtype=torch.float32, device=x.device) if shift is None else shift
    ws = torch.empty(lib().b200dm_bn_stats_workspace(c) // 4, dtype=torch.float32, device=x.device)
    check(lib().b200dm_bn_stats(ptr(x), x.numel() // c, c, ptr(gamma), ptr(beta), eps, ptr(scale), ptr(shift), ptr(ws), ws.numel() * 4,
                                stream()))
    return scale, shift


def make_norm_desc(x0, x1=None, kind=0, groups=1, act=None) -> L.NormDesc:
    d = L.NormDesc()
    d.voxels = int(np.prod(x0.shape[1:-1]))
    d.batch, d.c0, d.c1 = x0.shape[0], x0.shape[-1], (x1.shape[-1] if x1 is not None else 0)
    d.kind, d.groups, d.act, d.x_dtype, d.y_dtype = kind, groups, L.ACT[act], L.BF16, L.BF16
    return d


def gn_stats(x, groups, eps):
    L.check_storage(x)
    _dev()
    d = make_norm_desc(x, None, 1, groups)
    ws = torch.empty(lib().b200dm_gn_stats_workspace(C.byref(d)) // 4, dtype=torch.float32, device=x.device)
    mr = torch.empty(x.shape[0], groups, 2, dtype=torch.float32, device=x.device)
    check(lib().b200dm_gn_stats(C.byref(d), ptr(x), eps, ptr(mr), ptr(ws), ws.numel() * 4, stream()))
    return mr


def norm_act(x0, a, b, act=None, x1=None, kind=0, groups=1, mean_rstd=None, out=None):
    """y = act(affine(x)) over [x0, x1] concatenated on channels (16-bit in, 16-bit out)."""
    L.check_storage(x0, x1, out)
    _dev()
    d = make_norm_desc(x0, x1, kind, groups, act)
    if out is None:
        out = torch.empty(*x0.shape[:-1], d.c0 + d.c1, dtype=L.ACT_DTYPE, device=x0.device)
    check(lib().b200dm_norm_act_fwd(C.byref(d), ptr(x0), ptr(x1), ptr(a), ptr(b), ptr(mean_rstd), ptr(out), stream()))
    return out


def _ptr_array(ts):
    arr = (C.c_void_p * len(ts))()
    for i, t in enumerate(ts):
        arr[i] = t.data_ptr()
    return arr


def layernorm(x, gammas, betas, eps=1e-3):
    L.check_storage(x)
    _dev()
    c = x.shape[-1]
    rows = x.numel() // c
    ys = [torch.empty_like(x) for _ in gammas]
    check(lib().b200dm_layernorm_fwd(ptr(x), rows, c, eps, len(gammas), _ptr_array(gammas), _ptr_array(betas), _ptr_array(ys), stream()))
    return ys


def cast(x, dtype):
    _dev()
    y = torch.empty(x.shape, dtype=L.storage(dtype), device=x.device)
    check(lib().b200dm_cast(ptr(x), dt(x), ptr(y), dt(y), x.numel(), stream()))
    return y


# ------------------------------------------------------------------ K11 VQ
def vq_prepare(codebook_kd):
    _dev()
    sq = torch.empty(codebook_kd.shape[0], dtype=torch.float32, device=codebook_kd.device)
    check(lib().b200dm_vq_prepare(ptr(codebook_kd), codebook_kd.shape[0], codebook_kd.shape[1], ptr(sq), stream()))
    return sq


def vq_prepare_tc(codebook_kd, code_sqnorm):
    """Workspace of the tensor-core search (fp16 hi/lo halves of the codebook + scales), or None when (K, D) is outside its
    shapes (K % 128, D in {64,128,192,256})."""
    _dev()
    k, d = codebook_kd.shape
    nbytes = lib().b200dm_vq_tc_workspace_bytes(k, d)
    if nbytes == 0:
        return None
    ws = torch.empty((nbytes + 127) // 128 * 128, dtype=torch.uint8, device=codebook_kd.device)   # caching allocator: 512-byte aligned
    check(lib().b200dm_vq_prepare_tc(ptr(codebook_kd), ptr(code_sqnorm), k, d, ptr(ws), stream()))
    return ws


def vq_argmin_gather(x, codebook_kd, code_sqnorm=None, want_q=True, q_dtype=torch.float32, hist=None, tc_ws="auto", stats=None):
    """x (..., D) fp32|bf16; codebook (K, D) fp32 -> (idx int64 (N,), q (..., D) | None).  ``tc_ws``: workspace from
    vq_prepare_tc ('auto' builds it when the shape allows, None forces the fp32 SIMT kernel); both kernels return the same
    indices bit for bit."""
    _dev()
    D = x.shape[-1]
    n = x.numel() // D
    if code_sqnorm is None:
        code_sqnorm = vq_prepare(codebook_kd)
    if isinstance(tc_ws, str):
        tc_ws = vq_prepare_tc(codebook_kd, code_sqnorm)
    d = L.VqDesc()
    d.n, d.d, d.k, d.x_dtype, d.q_dtype = n, D, codebook_kd.shape[0], dt(x), (L.F32 if q_dtype == torch.float32 else L.BF16)
    idx = torch.empty(n, dtype=torch.int64, device=x.device)
    q = torch.empty(x.shape, dtype=L.storage(q_dtype), device=x.device) if want_q else None
    if tc_ws is not None and n > 0:
        check(lib().b200dm_vq_argmin_gather_tc(C.byref(d), ptr(x), ptr(codebook_kd), ptr(code_sqnorm), ptr(tc_ws), ptr(idx), ptr(q), ptr(hist),
                                               ptr(stats), stream()))
    else:
        check(lib().b200dm_vq_argmin_gather(C.byref(d), ptr(x), ptr(codebook_kd), ptr(code_sqnorm), ptr(idx), ptr(q), ptr(hist), stream()))
    return idx, q


# ------------------------------------------------------------------ K12 dense / softmax
def dense_f32(x, w, b=None, act_in=None, act_out=None):
    _dev()
    m, k = x.shape
    n = w.shape[1]
    y = torch.empty(m, n, dtype=torch.float32, device=x.device)
    check(lib().b200dm_dense_f32(ptr(x), ptr(w), ptr(b), ptr(y), m, k, n, L.ACT[act_in], L.ACT[act_out], stream()))
    return y


def softmax_rows(s, scale=1.0):
    _dev()
    cols = s.shape[-1]
    p = torch.empty(s.shape, dtype=L.ACT_DTYPE, device=s.device)
    check(lib().b200dm_softmax_rows(ptr(s), ptr(p), s.numel() // cols, cols, scale, stream()))
    return p


# ------------------------------------------------------------------ K1-K5 conv
def make_conv_desc(mode, batch, in_dhw, c0, c1, c_out, ksize=3, stride=1, act=None, post_act=None, y_dtype=torch.bfloat16,
                   chan_bias_rows=0, transposed_store=False, use_halo=False) -> L.ConvDesc:
    d = L.ConvDesc()
    d.mode, d.batch = mode, batch
    d.in_d, d.in_h, d.in_w = in_dhw
    d.c0, d.c1, d.c_out, d.ksize, d.stride = c0, c1, c_out, ksize, stride
    d.act, d.y_dtype = L.ACT[act], (L.F32 if y_dtype == torch.float32 else L.BF16)
    d.chan_bias_rows, d.use_halo = chan_bias_rows, int(use_halo)
    d.reserved[0], d.reserved[1] = L.ACT[post_act], int(transposed_store)
    return d


def pack_conv_weights(desc: L.ConvDesc, keras_kernel: torch.Tensor, transposed=False) -> torch.Tensor:
    """Keras kernel fp32 (k,k,k,Cin,Cout) [(k,k,k,Cout,Cin) if transposed] -> packed bf16 bytes (host)."""
    nbytes = lib().b200dm_conv_packed_weight_bytes(C.byref(desc))
    if nbytes == 0:
        raise L.B200dmError("pack_conv_weights: " + lib().b200dm_last_error().decode())
    w = keras_kernel.detach().to("cpu", torch.float32).contiguous()
    out = torch.empty(nbytes // 2, dtype=L.ACT_DTYPE)
    check(lib().b200dm_conv_pack_weights(C.byref(desc), C.c_void_p(w.data_ptr()), int(transposed), C.c_void_p(out.data_ptr())))
    return out


def fold_shortcut_weights(w_packed: torch.Tensor, sc_desc: L.ConvDesc, sc_packed: torch.Tensor) -> torch.Tensor:
    """Packed weights of a 3^3 conv with those of a 1^3 conv on the same output channels (``sc_desc``) appended to each row,
    zero-padded to a multiple of 3 k-blocks: the layout ``ConvPlan.set_shortcut`` reads."""
    kb = -(-sc_desc.c0 // 64) + -(-sc_desc.c1 // 64)
    rows = sc_packed.numel() // (kb * 64)
    pad = torch.zeros(rows, (-kb) % 3 * 64, dtype=w_packed.dtype, device=w_packed.device)
    return torch.cat([w_packed.view(rows, -1), sc_packed.to(w_packed.device).view(rows, -1), pad], dim=1).reshape(-1)


class ConvPlan:
    """One conv / GEMM invocation with fixed buffers (owns the TMA descriptors)."""

    def __init__(self, desc, x0, w_packed, y, x1=None, bias=None, chan_bias=None, t_dev=None, residual=None, prelu_alpha=None,
                 out_affine=None):
        L.check_storage(x0, x1, w_packed, residual, prelu_alpha, y)
        _dev()
        self.keep = (x0, x1, w_packed, bias, chan_bias, t_dev, residual, prelu_alpha, y) + tuple(out_affine or ())  # keep buffers alive
        # algorithmic HBM bytes of one launch: every operand read once, the output written once
        self.alg_bytes = float(sum(t.numel() * t.element_size() for t in (x0, x1, w_packed, residual, y) if t is not None))
        self.desc = desc
        h = C.c_void_p()
        check(lib().b200dm_conv_plan_create(C.byref(desc), ptr(x0), ptr(x1), ptr(w_packed), ptr(bias), ptr(chan_bias),
                                            ptr(t_dev), ptr(residual), ptr(prelu_alpha), ptr(y), C.byref(h)))
        self.h = h
        self.y = y
        self.owned = True
        if out_affine is not None:  # (scale, shift) of the consumer's folded BatchNorm
            check(lib().b200dm_conv_plan_set_out_affine(self.h, ptr(out_affine[0]), ptr(out_affine[1])))

    @property
    def flops(self):
        return lib().b200dm_conv_plan_flops(self.h)

    @property
    def info(self):
        halo, bn, ks = C.c_int32(), C.c_int32(), C.c_int32()
        check(lib().b200dm_conv_plan_info(self.h, C.byref(halo), C.byref(bn), C.byref(ks)))
        return dict(halo=halo.value, block_n=bn.value, ksplit=ks.value)   # halo: 0 per-tap GEMM, 1 halo kernel, 2 C_out=1 stencil

    def set_fused_update(self, upd_desc, x_t, x_prev, x_prev_16):
        """Output conv of the U-Net only: the epilogue applies the reverse-diffusion update to its eps tile and stores
        x_{t-1} (fp32 -> ``x_prev`` = ``x_t``, in place; 16-bit copy -> ``x_prev_16``) instead of eps.  False when the plan's
        kernel cannot (the caller then runs the stand-alone update kernel on the conv's eps output)."""
        rc = lib().b200dm_conv_plan_set_fused_update(self.h, C.byref(upd_desc), ptr(x_t), ptr(x_prev), ptr(x_prev_16))
        if rc == L.ERR_UNSUPPORTED:
            return False
        check(rc)
        self.keep = self.keep + (x_t, x_prev, x_prev_16, upd_desc)
        return True

    def set_shortcut(self, x0, x1, w_packed, bias):
        """Fold a 1^3 conv of [x0 | x1] into this 3^3 conv's K loop (a ResidualBlock's shortcut): ``w_packed`` from
        ``fold_shortcut_weights``, ``bias`` the two convs' biases summed.  False when the plan's kernel cannot (the caller then
        runs the 1^3 conv on its own and passes its output as the residual)."""
        rc = lib().b200dm_conv_plan_set_shortcut(self.h, x0.shape[-1], x1.shape[-1] if x1 is not None else 0, ptr(x0), ptr(x1),
                                                 ptr(w_packed), ptr(bias))
        if rc == L.ERR_UNSUPPORTED:
            return False
        check(rc)
        nbytes = lambda t: float(t.numel() * t.element_size()) if t is not None else 0.0  # noqa: E731
        self.alg_bytes += nbytes(x0) + nbytes(x1) + nbytes(w_packed) - nbytes(self.keep[2])
        self.keep = self.keep + (x0, x1, w_packed, bias)
        return True

    def run(self):
        check(lib().b200dm_conv_plan_run(self.h, stream()))
        return self.y

    def gn_partials(self):
        """GroupNorm partial sums as a by-product of this conv: -> (workspace fp64 (B * rows, C, 2), rows per sample), or None
        when the plan's kernel cannot produce them (the caller then runs a statistics pass over y)."""
        rows = C.c_int32(0)
        nbytes = lib().b200dm_conv_plan_gn_partials_bytes(self.h, C.byref(rows))
        if nbytes == 0:
            return None
        ws = torch.zeros(nbytes // 8, dtype=torch.float64, device=self.y.device)
        check(lib().b200dm_conv_plan_set_gn_partials(self.h, ptr(ws), nbytes))
        self.keep = self.keep + (ws,)
        return ws, rows.value

    def release(self):  # ownership moved into a program
        self.owned = False

    def __del__(self):
        try:
            if getattr(self, "owned", False) and self.h:
                lib().b200dm_conv_plan_destroy(self.h)
                self.h = None
        except Exception:  # interpreter shutdown
            pass


def conv_out_shape(mode, in_dhw, stride):
    if mode == L.CONV_PARITY:
        return tuple(2 * s for s in in_dhw)
    return tuple(-(-s // stride) for s in in_dhw)


def conv3d(x0, keras_kernel, bias=None, x1=None, mode=L.CONV_DIRECT, stride=1, act=None, post_act=None, residual=None,
           chan_bias=None, prelu_alpha=None, y_dtype=torch.bfloat16, transposed=False, out_affine=None, use_halo=False):
    """Convenience one-shot conv (tests): packs, plans, runs.  x bf16 NDHWC; returns y NDHWC."""
    dev = _dev()
    B, D, H, W, c0 = x0.shape
    c1 = x1.shape[-1] if x1 is not None else 0
    k = keras_kernel.shape[0]
    c_out = keras_kernel.shape[3] if transposed else keras_kernel.shape[4]
    desc = make_conv_desc(mode, B, (D, H, W), c0, c1, c_out, k, stride, act, post_act, y_dtype,
                          chan_bias_rows=B if chan_bias is not None else 0, use_halo=use_halo)
    wp = pack_conv_weights(desc, keras_kernel, transposed).to(dev)
    od, oh, ow = conv_out_shape(mode, (D, H, W), stride)
    y = torch.empty(B, od, oh, ow, c_out, dtype=L.storage(y_dtype), device=dev)
    plan = ConvPlan(desc, x0, wp, y, x1=x1, bias=bias, chan_bias=chan_bias, residual=residual, prelu_alpha=prelu_alpha,
                    out_affine=out_affine)
    plan.run()
    return y


def batched_gemm(a, b, y_dtype=torch.float32, residual=None):
    """y[n] = a[n] (M,K) @ b[n] (N,K)^T, 16-bit operands, fp32 accumulate (attention matmuls)."""
    L.check_storage(a, b, residual)
    dev = _dev()
    B, M, K = a.shape
    N = b.shape[1]
    desc = make_conv_desc(L.CONV_BATCHED_GEMM, B, (1, 1, M), K, 0, N, 1, 1, None, None, y_dtype)
    y = torch.empty(B, M, N, dtype=L.storage(y_dtype), device=dev)
    plan = ConvPlan(desc, a, b, y, residual=residual)
    plan.run()
    return y


# ------------------------------------------------------------------ K8/K9 flash attention
class AttnPlan:
    """softmax(scale * q k^T) v (+ residual) with fixed buffers: q (B,Lq,D), k (B,Lk,D), vt (B,D,Lk), o (B,Lq,D), bf16."""

    def __init__(self, q, k, vt, o, scale, residual=None):
        """q / k may be column blocks of a wider (B, L, ld) tensor (views ``t[..., a:a+D]``): their row stride goes into the desc."""
        _dev()
        B, Lq, D = q.shape
        Lk = k.shape[1]
        assert tuple(k.shape) == (B, Lk, D) and tuple(vt.shape) == (B, D, Lk) and tuple(o.shape) == (B, Lq, D)
        assert all(t.dtype == L.ACT_DTYPE for t in (q, k, vt, o)) and vt.is_contiguous() and o.is_contiguous()
        for t, L_ in ((q, Lq), (k, Lk)):   # rows of D contiguous elements, uniform row stride, samples L rows apart
            assert t.stride(2) == 1 and t.stride(0) == L_ * t.stride(1), "q / k: unsupported layout"
        self.keep = (q, k, vt, o, residual)
        d = L.AttnDesc()
        d.batch, d.lq, d.lk, d.d, d.scale = B, Lq, Lk, D, float(scale)
        d.reserved[0] = 0 if q.stride(1) == D else q.stride(1)
        d.reserved[1] = 0 if k.stride(1) == D else k.stride(1)
        h = C.c_void_p()
        check(lib().b200dm_attention_plan_create(C.byref(d), ptr(q), ptr(k), ptr(vt), ptr(residual), ptr(o), C.byref(h)))
        self.h, self.o, self.owned = h, o, True

    @property
    def flops(self):
        return lib().b200dm_attention_plan_flops(self.h)

    def run(self):
        check(lib().b200dm_attention_plan_run(self.h, stream()))
        return self.o

    def release(self):
        self.owned = False

    def __del__(self):
        try:
            if getattr(self, "owned", False) and self.h:
                lib().b200dm_attention_plan_destroy(self.h)
                self.h = None
        except Exception:
            pass


def attention(q, k, vt, scale, residual=None):
    """One-shot flash attention (tests): returns o (B,Lq,D) bf16."""
    o = torch.empty(q.shape, dtype=q.dtype, device=q.device)
    AttnPlan(q, k, vt, o, scale, residual).run()
    return o
