"""First stage on the sm_100a kernels: VQ codebook quantizer + 3D decoders (latents -> MRI volumes).

Mirrors the attribute surface the reference's DiffusionModel uses (``.encoder / .quantizer / .decoder``):
    VectorQuantizer            networks/vqvae3d_monai.py:112-177 (codebook (D,K)); vqgan_attn_cp.py:140-247 ((K,D))
    MonaiDecoder  (family D1)  networks/vqvae3d_monai.py:309-391 + VQVAEResidualUnit :218-234
    AttnCpDecoder (family D5)  networks/vqgan_attn_cp.py:339-427 + VQVAEResidualUnit :250-276
    VQVAE / VQGAN              networks/vqvae3d_monai.py:394-457 / vqgan_attn_cp.py:569-590 (constructor surface)
    MonaiEncoder  (8f.2)       networks/vqvae3d_monai.py:237-306 (volumes -> pre-quantisation latents; front half of train_step)
The other families' encoders are not built: their ``.encoder`` raises.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import _lib as L
from . import ops
from .program import Program
from . import weights as Wt


# ================================================================== quantizer
class VectorQuantizer:
    """``layout`` 'DK': embeddings stored (embedding_dim, num_embeddings) like vqvae3d_monai/vqgan;
    'KD': (num_embeddings, embedding_dim) like vqgan_gnorm/stride/attn_cp."""

    def __init__(self, num_embeddings, embedding_dim, beta=0.25, layout="DK", seed=3):
        self.num_embeddings, self.embedding_dim, self.beta, self.layout = num_embeddings, embedding_dim, beta, layout
        rng = np.random.default_rng(seed)
        if layout == "DK":   # HeUniform on (D,K): limit sqrt(6/fan_in), fan_in = D (vqvae3d_monai.py:123-127)
            lim = np.sqrt(6.0 / embedding_dim)
            e = rng.uniform(-lim, lim, size=(embedding_dim, num_embeddings))
        else:                # tf.random_uniform_initializer() = U(-0.05, 0.05) (vqgan_attn_cp.py:154-158)
            e = rng.uniform(-0.05, 0.05, size=(num_embeddings, embedding_dim))
        self.embeddings = torch.from_numpy(e.astype(np.float32))
        self.codebooks_used = torch.zeros(num_embeddings, dtype=torch.int32)
        self._dev = None

    def set_embeddings(self, e):
        e = torch.as_tensor(e).float().cpu()
        want = (self.embedding_dim, self.num_embeddings) if self.layout == "DK" else (self.num_embeddings, self.embedding_dim)
        if tuple(e.shape) != want:
            raise ValueError(f"codebook: expected {want} ({self.layout} layout), got {tuple(e.shape)}")
        self.embeddings, self._dev = e, None

    def _device_state(self):
        if self._dev is None:
            L.require_gpu()
            dev = torch.device("cuda", torch.cuda.current_device())
            kd = (self.embeddings.t() if self.layout == "DK" else self.embeddings).contiguous().to(dev)
            sq = ops.vq_prepare(kd)
            self._dev = dict(kd=kd, sq=sq, tc=ops.vq_prepare_tc(kd, sq), hist=torch.zeros(self.num_embeddings, dtype=torch.int32, device=dev))
        return self._dev

    def get_code_indices(self, flattened_inputs, distribution=False):
        """(N, D) -> (N,) int64; lowest index on ties.  ``distribution=True`` returns the (N, K) fp32 squared-distance matrix
        instead (the reference's training-time diagnostic, vqvae3d_monai.py:172-175)."""
        st = self._device_state()
        if distribution:   # the (N, K) squared-distance matrix itself (vqvae3d_monai.py:172-175), same fp32 arithmetic as the argmin
            x = flattened_inputs.contiguous()
            d = L.VqDesc()
            d.n, d.d, d.k, d.x_dtype, d.q_dtype = x.shape[0], x.shape[1], self.num_embeddings, L.dt(x), L.F32
            dist = torch.empty(x.shape[0], self.num_embeddings, dtype=torch.float32, device=x.device)
            L.check(L.lib().b200dm_vq_distances(d, L.ptr(x), L.ptr(st["kd"]), L.ptr(st["sq"]), L.ptr(dist), L.stream()))
            return dist
        idx, _ = ops.vq_argmin_gather(flattened_inputs.contiguous(), st["kd"], st["sq"], want_q=False, tc_ws=st["tc"])
        return idx

    def quantize(self, x, q_dtype=torch.float32):
        """-> (quantized like x, indices (N,), perplexity).  Returns the gathered code rows q; the reference's
        straight-through form x + (q - x) equals q up to 1 ulp (SURVEY Q2)."""
        st = self._device_state()
        st["hist"].zero_()
        idx, q = ops.vq_argmin_gather(x.contiguous(), st["kd"], st["sq"], want_q=True, q_dtype=q_dtype, hist=st["hist"], tc_ws=st["tc"])
        counts = st["hist"].cpu()
        self.codebooks_used += counts                       # codebooks_used.assign_add (vqvae3d_monai.py:161)
        p = counts.double() / max(1, idx.numel())
        perplexity = float(torch.exp(-(p * torch.log(p + 1e-10)).sum()))
        return q, idx, perplexity

    def __call__(self, x):
        q, _, perplexity = self.quantize(x)
        return q, perplexity


# ================================================================== decoders
class _DecoderBase:
    spec: list
    out_channels: int

    def __init__(self):
        self._params = None   # random-initialised lazily (per-voxel PReLU alphas make D1 large)
        self.prog = None

    @property
    def params(self):
        if self._params is None:
            self._params = Wt.init_params(self.spec, seed=1, mode="keras")
        return self._params

    def set_weights(self, params):
        Wt.check_against_spec(params, self.spec)
        self._params = {k: torch.as_tensor(v).float().cpu() for k, v in params.items()}
        self.prog = None

    def count_params(self):
        return sum(int(np.prod(s)) for _, s, _ in self.spec)

    def _conv(self, pr, x0, kernel, bias, cout, k=3, mode=L.CONV_DIRECT, act=None, post_act=None, residual=None,
              prelu_alpha=None, y_dtype=torch.bfloat16, transposed=False, note="", stride=1):
        B, D, H, W, c0 = x0.shape
        desc = ops.make_conv_desc(mode, B, (D, H, W), c0, 0, cout, k, stride, act, post_act, y_dtype)
        wp = ops.pack_conv_weights(desc, kernel, transposed).to(self.device)
        od, oh, ow = ops.conv_out_shape(mode, (D, H, W), stride)
        y = pr.buf((B, od, oh, ow, cout), y_dtype)
        return pr.conv(desc, x0, wp, y, bias=bias.to(self.device).contiguous(), residual=residual,
                       prelu_alpha=prelu_alpha, note=note)

    def __call__(self, latents):
        """decoder(latents (B,s,s,s,D) fp32|bf16) -> volumes (B,S,S,S,out) fp32."""
        if self.prog is None or tuple(latents.shape) != tuple(self.z_in.shape):
            self.compile(latents.shape[0], latents.shape[1])
        z = latents.to(self.device)
        self.z_in.copy_(z if z.dtype == L.ACT_DTYPE else ops.cast(z.contiguous().float(), L.ACT_DTYPE))
        self.prog.run()
        return self.out.clone()


class MonaiDecoder(_DecoderBase):
    """Conv3(D->c_top) PReLU; per level: R x [relu(x + PReLU(BN(Conv3(relu(Conv3(x))))))], ConvT(k4,s2) (+ReLU)."""

    def __init__(self, in_channels, out_channels, num_channels, num_res_layers, num_res_channels, in_size,
                 upsample_parameters=None, dropout=None, output_act=None, kernel_resize=False):
        self.cin, self.out_channels, self.R, self.in_size = in_channels, out_channels, num_res_layers, in_size
        self.ch, self.rch = list(reversed(num_channels)), list(reversed(num_res_channels))
        self.output_act = output_act
        sp, s = [], in_size
        c = self.ch[0]
        sp += [("stem.kernel", (3, 3, 3, in_channels, c), "glorot"), ("stem.bias", (c,), "zeros"), ("stem.prelu.alpha", (s, s, s, c), "zeros")]
        for i, c in enumerate(self.ch):
            for j in range(self.R):
                n, rc = f"level.{i}.res.{j}", self.rch[i]
                sp += [(f"{n}.conv1.kernel", (3, 3, 3, c, rc), "glorot"), (f"{n}.conv1.bias", (rc,), "zeros"),
                       (f"{n}.conv2.kernel", (3, 3, 3, rc, c), "glorot"), (f"{n}.conv2.bias", (c,), "zeros"),
                       (f"{n}.norm.gamma", (c,), "ones"), (f"{n}.norm.beta", (c,), "zeros"),
                       (f"{n}.norm.mean", (c,), "zeros"), (f"{n}.norm.var", (c,), "ones"),
                       (f"{n}.prelu.alpha", (s, s, s, c), "zeros")]
            out = out_channels if i == len(self.ch) - 1 else self.ch[i + 1]
            sp += [(f"level.{i}.up.kernel", (4, 4, 4, out, c), "glorot"), (f"level.{i}.up.bias", (out,), "zeros")]
            s *= 2
        self.spec = sp
        super().__init__()

    def compile(self, batch, in_size=None):
        L.require_gpu()
        assert in_size in (None, self.in_size), "per-voxel PReLU alphas lock the decoder to its build resolution"
        P = self.params
        self.device = dev = torch.device("cuda", torch.cuda.current_device())
        pr = self.prog = Program(dev)
        s = self.in_size
        self.z_in = pr.buf((batch, s, s, s, self.cin))
        alpha = lambda n: P[n].to(dev, L.ACT_DTYPE).contiguous()  # noqa: E731
        x = self._conv(pr, self.z_in, P["stem.kernel"], P["stem.bias"], self.ch[0], prelu_alpha=alpha("stem.prelu.alpha"), note="stem")
        for i, c in enumerate(self.ch):
            for j in range(self.R):
                n = f"level.{i}.res.{j}"
                h = self._conv(pr, x, P[f"{n}.conv1.kernel"], P[f"{n}.conv1.bias"], self.rch[i], act="relu", note=f"{n}.conv1")
                # BN (inference, eps 1e-3) folded into conv2: w' = w*scale[co], b' = b*scale + shift
                scale = P[f"{n}.norm.gamma"] * torch.rsqrt(P[f"{n}.norm.var"] + 1e-3)
                shift = P[f"{n}.norm.beta"] - P[f"{n}.norm.mean"] * scale
                x = self._conv(pr, h, P[f"{n}.conv2.kernel"] * scale, P[f"{n}.conv2.bias"] * scale + shift, c,
                               prelu_alpha=alpha(f"{n}.prelu.alpha"), residual=x, post_act="relu", note=f"{n}.conv2")
            last = i == len(self.ch) - 1
            out = self.out_channels if last else self.ch[i + 1]
            act = "relu" if (not last or self.output_act) else None
            x = self._conv(pr, x, P[f"level.{i}.up.kernel"], P[f"level.{i}.up.bias"], out, k=4, mode=L.CONV_PARITY, act=act,
                           y_dtype=torch.float32 if last else torch.bfloat16, transposed=True, note=f"level.{i}.up")
        self.out = x
        torch.cuda.synchronize(dev)
        return self


class MonaiEncoder(_DecoderBase):
    """vqvae3d_monai.Encoder (:237-306): per level Conv3D(c_i, k4, s2, 'same') ReLU, R x VQVAEResidualUnit; Conv3(->D) PReLU.
    volumes (B,S,S,S,in) -> pre-quantisation latents (B,s,s,s,D) fp32, s = S / 2^levels.  The input's channels are zero-padded
    to 8 (one 16-byte NDHWC vector) together with the first kernel's C_in."""

    def __init__(self, in_channels, out_channels, num_channels, num_res_layers, num_res_channels, in_size,
                 downsample_parameters=None, dropout=None):
        self.cin, self.out_channels, self.R, self.in_size = in_channels, out_channels, num_res_layers, in_size
        self.ch, self.rch = list(num_channels), list(num_res_channels)
        if downsample_parameters is not None:
            for dp in downsample_parameters:
                if tuple(dp[:3]) != (2, 4, 1) or dp[3] not in ("same", 1):
                    raise NotImplementedError(f"downsample_parameters {dp}: only (stride 2, kernel 4, dilation 1, 'same') is built")
        sp, s, cin = [], in_size, in_channels
        for i, c in enumerate(self.ch):
            s //= 2
            sp += [(f"level.{i}.down.kernel", (4, 4, 4, cin, c), "glorot"), (f"level.{i}.down.bias", (c,), "zeros")]
            for j in range(self.R):
                n, rc = f"level.{i}.res.{j}", self.rch[i]
                sp += [(f"{n}.conv1.kernel", (3, 3, 3, c, rc), "glorot"), (f"{n}.conv1.bias", (rc,), "zeros"),
                       (f"{n}.conv2.kernel", (3, 3, 3, rc, c), "glorot"), (f"{n}.conv2.bias", (c,), "zeros"),
                       (f"{n}.norm.gamma", (c,), "ones"), (f"{n}.norm.beta", (c,), "zeros"),
                       (f"{n}.norm.mean", (c,), "zeros"), (f"{n}.norm.var", (c,), "ones"),
                       (f"{n}.prelu.alpha", (s, s, s, c), "zeros")]
            cin = c
        sp += [("head.kernel", (3, 3, 3, cin, out_channels), "glorot"), ("head.bias", (out_channels,), "zeros"),
               ("head.prelu.alpha", (s, s, s, out_channels), "zeros")]
        self.spec = sp
        super().__init__()

    def compile(self, batch, in_size=None):
        L.require_gpu()
        assert in_size in (None, self.in_size), "per-voxel PReLU alphas lock the encoder to its build resolution"
        P = self.params
        self.device = dev = torch.device("cuda", torch.cuda.current_device())
        pr = self.prog = Program(dev)
        S = self.in_size
        cpad = -(-self.cin // 8) * 8
        self.z_in = pr.buf((batch, S, S, S, cpad))
        self.z_in.zero_()
        alpha = lambda n: P[n].to(dev, L.ACT_DTYPE).contiguous()  # noqa: E731
        x = self.z_in
        for i, c in enumerate(self.ch):
            w = P[f"level.{i}.down.kernel"]
            if i == 0 and cpad != self.cin:
                w = torch.cat([w, torch.zeros(4, 4, 4, cpad - self.cin, c)], dim=3)
            x = self._conv(pr, x, w, P[f"level.{i}.down.bias"], c, k=4, stride=2, act="relu", note=f"level.{i}.down")
            for j in range(self.R):
                n = f"level.{i}.res.{j}"
                h = self._conv(pr, x, P[f"{n}.conv1.kernel"], P[f"{n}.conv1.bias"], self.rch[i], act="relu", note=f"{n}.conv1")
                scale = P[f"{n}.norm.gamma"] * torch.rsqrt(P[f"{n}.norm.var"] + 1e-3)   # BN (inference) folded into conv2
                shift = P[f"{n}.norm.beta"] - P[f"{n}.norm.mean"] * scale
                x = self._conv(pr, h, P[f"{n}.conv2.kernel"] * scale, P[f"{n}.conv2.bias"] * scale + shift, c,
                               prelu_alpha=alpha(f"{n}.prelu.alpha"), residual=x, post_act="relu", note=f"{n}.conv2")
        self.out = self._conv(pr, x, P["head.kernel"], P["head.bias"], self.out_channels, prelu_alpha=alpha("head.prelu.alpha"),
                              y_dtype=torch.float32, note="head")
        torch.cuda.synchronize(dev)
        return self

    def __call__(self, volumes):
        """encoder(volumes (B,S,S,S,in) fp32|bf16) -> latents (B,s,s,s,D) fp32."""
        if getattr(self, "weights_missing", None):
            raise L.B200dmError(f"encoder: {self.weights_missing} holds no encoder tensors -- encode() would run on random weights")
        if self.prog is None or volumes.shape[0] != self.z_in.shape[0]:
            self.compile(volumes.shape[0], volumes.shape[1])
        v = volumes.to(self.device)
        self.z_in[..., :self.cin].copy_(v if v.dtype == L.ACT_DTYPE else ops.cast(v.contiguous().float(), L.ACT_DTYPE))
        self.prog.run()
        return self.out.clone()


class AttnCpDecoder(_DecoderBase):
    """Conv1(D->c_top) GN(min(D,32)) SiLU; [ConvT(k4,s2,c_i), 2 x (GN SiLU Conv3 GN SiLU Conv3 + x)] x (L-1); Conv3(->out)."""

    def __init__(self, in_channels, out_channels, num_channels, **_unused):
        self.cin, self.out_channels = in_channels, out_channels
        self.ch = list(reversed(num_channels))
        c0 = self.ch[0]
        sp = [("stem.kernel", (1, 1, 1, in_channels, c0), "glorot"), ("stem.bias", (c0,), "zeros"),
              ("stem.norm.gamma", (c0,), "ones"), ("stem.norm.beta", (c0,), "zeros")]
        for i in range(1, len(self.ch)):
            c = self.ch[i]
            sp += [(f"level.{i}.up.kernel", (4, 4, 4, c, self.ch[i - 1]), "glorot"), (f"level.{i}.up.bias", (c,), "zeros")]
            for j in range(2):
                n = f"level.{i}.res.{j}"
                sp += [(f"{n}.norm1.gamma", (c,), "ones"), (f"{n}.norm1.beta", (c,), "zeros"),
                       (f"{n}.conv1.kernel", (3, 3, 3, c, c), "glorot"), (f"{n}.conv1.bias", (c,), "zeros"),
                       (f"{n}.norm2.gamma", (c,), "ones"), (f"{n}.norm2.beta", (c,), "zeros"),
                       (f"{n}.conv2.kernel", (3, 3, 3, c, c), "glorot"), (f"{n}.conv2.bias", (c,), "zeros")]
        sp += [("head.kernel", (3, 3, 3, self.ch[-1], out_channels), "glorot"), ("head.bias", (out_channels,), "zeros")]
        self.spec = sp
        super().__init__()

    def compile(self, batch, in_size):
        L.require_gpu()
        P = self.params
        self.device = dev = torch.device("cuda", torch.cuda.current_device())
        pr = self.prog = Program(dev)
        s = in_size
        self.z_in = pr.buf((batch, s, s, s, self.cin))
        g = lambda n: P[n].to(dev).contiguous()  # noqa: E731

        def gn_silu(x, name, groups):
            mr = pr.gn_stats(x, groups, 1e-6, note=f"{name}.stats")
            return pr.norm_act(x, g(f"{name}.gamma"), g(f"{name}.beta"), pr.buf(x.shape), act="silu", kind=1, groups=groups,
                               mean_rstd=mr, note=name)

        x = self._conv(pr, self.z_in, P["stem.kernel"], P["stem.bias"], self.ch[0], k=1, note="stem")
        x = gn_silu(x, "stem.norm", min(self.cin, 32))
        for i in range(1, len(self.ch)):
            c = self.ch[i]
            grp = min(c, 32)
            x = self._conv(pr, x, P[f"level.{i}.up.kernel"], P[f"level.{i}.up.bias"], c, k=4, mode=L.CONV_PARITY, transposed=True,
                           note=f"level.{i}.up")
            def norm_conv(t, norm, conv, residual=None):
                """Conv3(SiLU(GN(t))) (vqgan_attn_cp.py:262-270) = GroupNorm statistics (from the producing conv's epilogue when its
                kernel accumulates them) -> fused GN + SiLU pass -> conv.  (Normalising the slabs inside the d-sweeping conv instead
                of the pass measured slower: 3.0 ms against 1.61 + 0.72 ms at 128^3, B=16.)"""
                return self._conv(pr, gn_silu(t, norm, grp), P[f"{conv}.kernel"], P[f"{conv}.bias"], c, residual=residual, note=conv)

            for j in range(2):
                n = f"level.{i}.res.{j}"
                h = norm_conv(x, f"{n}.norm1", f"{n}.conv1")
                x = norm_conv(h, f"{n}.norm2", f"{n}.conv2", residual=x)
        self.out = self._conv(pr, x, P["head.kernel"], P["head.bias"], self.out_channels, y_dtype=torch.float32, note="head")
        torch.cuda.synchronize(dev)
        return self


class VqganFamilyDecoder(_DecoderBase):
    """Decoders D2 / D3 / D4 (act_fn='prelu'):  'vqgan' networks/vqgan.py:378-475, 'gnorm' vqgan_gnorm.py:382-484,
    'stride' vqgan_stride.py:376-480 (residual units :256-286 of each file).

      stem   Conv3 -> [BN | GN(8,1e-6) | -] -> PReLU
      level  R x relu(x + PReLU(Norm(Conv3(relu(Conv3 x)))))
             'vqgan'/'gnorm': ConvT(k4,s2) -> [BN | GN] (-> PReLU unless last)
             'stride':        Conv3D(k4,s1,'same') -> UpSampling3D(2) -> [GN(out/2,1e-6) if out<32] (-> PReLU unless last)
    BatchNorm (inference) is folded into the preceding conv's weights; GroupNorm runs as statistics + one fused
    norm -> PReLU -> +residual -> ReLU pass; the up-sampling is folded into that pass's read."""

    def __init__(self, variant, in_channels, out_channels, num_channels, num_res_layers, num_res_channels, in_size,
                 output_act=None):
        assert variant in ("vqgan", "gnorm", "stride")
        self.variant, self.cin, self.out_channels, self.R, self.in_size = variant, in_channels, out_channels, num_res_layers, in_size
        self.ch, self.rch = list(reversed(num_channels)), list(reversed(num_res_channels))
        self.output_act = output_act
        s, c = in_size, self.ch[0]
        sp = [("stem.kernel", (3, 3, 3, in_channels, c), "glorot"), ("stem.bias", (c,), "zeros")]
        sp += self._norm_spec("stem.norm", self._stem_norm()[0], c) + [("stem.prelu.alpha", (s, s, s, c), "zeros")]
        for i, c in enumerate(self.ch):
            for j in range(self.R):
                n, rc = f"level.{i}.res.{j}", self.rch[i]
                sp += [(f"{n}.conv1.kernel", (3, 3, 3, c, rc), "glorot"), (f"{n}.conv1.bias", (rc,), "zeros"),
                       (f"{n}.conv2.kernel", (3, 3, 3, rc, c), "glorot"), (f"{n}.conv2.bias", (c,), "zeros")]
                sp += self._norm_spec(f"{n}.norm", self._res_norm(c)[0], c) + [(f"{n}.prelu.alpha", (s, s, s, c), "zeros")]
            last = i == len(self.ch) - 1
            out = out_channels if last else self.ch[i + 1]
            sp += [(f"level.{i}.up.kernel", (4, 4, 4, c, out) if variant == "stride" else (4, 4, 4, out, c), "glorot"),
                   (f"level.{i}.up.bias", (out,), "zeros")]
            s *= 2
            sp += self._norm_spec(f"level.{i}.up.norm", self._up_norm(out)[0], out)
            if not last:
                sp += [(f"level.{i}.up.prelu.alpha", (s, s, s, out), "zeros")]
        self.spec = sp
        super().__init__()

    # (kind, groups, eps) per site, as written in the reference files
    def _stem_norm(self):
        return {"vqgan": ("bn", 0, 1e-3), "gnorm": ("gn", 8, 1e-6), "stride": (None, 0, 0.0)}[self.variant]

    def _res_norm(self, c):
        if self.variant == "gnorm":
            return ("gn", 1, 1e-3) if c == 2 else ("gn", 8, 1e-6)
        return ("bn", 0, 1e-3)

    def _up_norm(self, out):
        if self.variant == "vqgan":
            return ("bn", 0, 1e-3)
        if self.variant == "gnorm":
            return ("gn", int(out / 2), 1e-3) if out < 32 else ("gn", 8, 1e-6)
        return ("gn", int(out / 2), 1e-6) if out < 32 else (None, 0, 0.0)

    @staticmethod
    def _norm_spec(name, kind, c):
        if kind is None:
            return []
        sp = [(f"{name}.gamma", (c,), "ones"), (f"{name}.beta", (c,), "zeros")]
        return sp + ([(f"{name}.mean", (c,), "zeros"), (f"{name}.var", (c,), "ones")] if kind == "bn" else [])

    def compile(self, batch, in_size=None):
        L.require_gpu()
        assert in_size in (None, self.in_size), "per-voxel PReLU alphas lock the decoder to its build resolution"
        P = self.params
        self.device = dev = torch.device("cuda", torch.cuda.current_device())
        pr = self.prog = Program(dev)
        s = self.in_size
        self.z_in = pr.buf((batch, s, s, s, self.cin))
        alpha = lambda n: P[n].to(dev, L.ACT_DTYPE).contiguous()  # noqa: E731
        g = lambda n: P[n].to(dev).contiguous()  # noqa: E731

        def bn_fold(name, kernel, bias, eps, transposed=False):
            """conv -> BN(inference) == conv with w' = w * scale[co], b' = b * scale + shift."""
            scale = P[f"{name}.gamma"] * torch.rsqrt(P[f"{name}.var"] + eps)
            shift = P[f"{name}.beta"] - P[f"{name}.mean"] * scale
            k = kernel * (scale.view(1, 1, 1, -1, 1) if transposed else scale)
            return k, bias * scale + shift

        def gn_apply(h, name, groups, eps, y, **kw):
            """GroupNorm statistics of h (taken BEFORE any up-sampling) + the fused apply pass into y."""
            if groups < 1:
                raise ValueError(f"{name}: GroupNormalization(groups={groups}) -- the reference layer cannot be built either")
            if h.dtype == torch.float32:
                if groups != 1:
                    raise L.B200dmError(f"{name}: fp32 group norm supports one group (the 1-2 channel network output)")
                mr = pr.stats_f32(h, eps, note=f"{name}.stats")
            else:
                mr = pr.gn_stats(h, groups, eps, note=f"{name}.stats")
            return pr.norm_act_ex(h, g(f"{name}.gamma"), g(f"{name}.beta"), y, kind=1, groups=groups, mean_rstd=mr, note=name, **kw)

        c = self.ch[0]
        kind, groups, eps = self._stem_norm()
        if kind == "bn":
            k, b = bn_fold("stem.norm", P["stem.kernel"], P["stem.bias"], eps)
            x = self._conv(pr, self.z_in, k, b, c, prelu_alpha=alpha("stem.prelu.alpha"), note="stem")
        elif kind == "gn":
            h = self._conv(pr, self.z_in, P["stem.kernel"], P["stem.bias"], c, note="stem")
            x = gn_apply(h, "stem.norm", groups, eps, pr.buf(h.shape), prelu_alpha=alpha("stem.prelu.alpha"))
        else:
            x = self._conv(pr, self.z_in, P["stem.kernel"], P["stem.bias"], c, prelu_alpha=alpha("stem.prelu.alpha"), note="stem")
        for i, c in enumerate(self.ch):
            for j in range(self.R):
                n = f"level.{i}.res.{j}"
                h = self._conv(pr, x, P[f"{n}.conv1.kernel"], P[f"{n}.conv1.bias"], self.rch[i], act="relu", note=f"{n}.conv1")
                kind, groups, eps = self._res_norm(c)
                if kind == "bn":
                    k, b = bn_fold(f"{n}.norm", P[f"{n}.conv2.kernel"], P[f"{n}.conv2.bias"], eps)
                    x = self._conv(pr, h, k, b, c, prelu_alpha=alpha(f"{n}.prelu.alpha"), residual=x, post_act="relu", note=f"{n}.conv2")
                else:
                    h = self._conv(pr, h, P[f"{n}.conv2.kernel"], P[f"{n}.conv2.bias"], c, note=f"{n}.conv2")
                    x = gn_apply(h, f"{n}.norm", groups, eps, pr.buf(h.shape), prelu_alpha=alpha(f"{n}.prelu.alpha"), residual=x,
                                 post_act="relu")
            last = i == len(self.ch) - 1
            out = self.out_channels if last else self.ch[i + 1]
            n = f"level.{i}.up"
            kind, groups, eps = self._up_norm(out)
            pa = None if last else alpha(f"{n}.prelu.alpha")
            final_act = "relu" if (last and self.output_act) else None
            y_dtype = torch.float32 if last else torch.bfloat16
            B_, D_ = x.shape[0], x.shape[1]
            if self.variant == "stride":
                # Conv3D(k=4, s=1, 'same') at low resolution, then ONE pass: nearest x2 + [GN] + [PReLU]
                h = self._conv(pr, x, P[f"{n}.kernel"], P[f"{n}.bias"], out, k=4, y_dtype=y_dtype, note=n)
                y = pr.buf((B_, 2 * D_, 2 * D_, 2 * D_, out), y_dtype)
                if kind == "gn":
                    x = gn_apply(h, f"{n}.norm", groups, eps, y, prelu_alpha=pa, act=final_act, upsample=True)
                else:
                    one, zero = torch.ones(out, device=dev), torch.zeros(out, device=dev)
                    x = pr.norm_act_ex(h, one, zero, y, prelu_alpha=pa, act=final_act, upsample=True, note=f"{n}.upsample")
            elif kind == "bn":
                k, b = bn_fold(f"{n}.norm", P[f"{n}.kernel"], P[f"{n}.bias"], eps, transposed=True)
                x = self._conv(pr, x, k, b, out, k=4, mode=L.CONV_PARITY, prelu_alpha=pa, act=final_act, y_dtype=y_dtype,
                               transposed=True, note=n)
            else:
                h = self._conv(pr, x, P[f"{n}.kernel"], P[f"{n}.bias"], out, k=4, mode=L.CONV_PARITY, y_dtype=y_dtype, transposed=True, note=n)
                x = gn_apply(h, f"{n}.norm", groups, eps, pr.buf(h.shape, y_dtype), prelu_alpha=pa, act=final_act)
        self.out = x
        torch.cuda.synchronize(dev)
        return self


# ================================================================== model wrappers (constructor surface)
class _NoEncoder:
    def __call__(self, *a, **k):
        raise NotImplementedError("the encoder is not on the sampling/decode hot path (SURVEY section 8f.2); not built")


class VQVAE:
    """networks/vqvae3d_monai.VQVAE constructor surface; ``latent_size`` (build addition) sizes the per-voxel PReLUs
    (Keras infers it from the fixed 128^3 input: 128 / 2^levels)."""

    def __init__(self, in_channels, out_channels, num_channels, num_res_layers, num_res_channels,
                 downsample_parameters=((2, 4, 1, 1),) * 3, upsample_parameters=((2, 4, 1, 1, 0),) * 3,
                 num_embeddings=128, embedding_dim=64, dropout=0.1, act="relu", output_act=None, num_gpus=2,
                 kernel_resize=False, latent_size=None):
        self.in_channels, self.out_channels, self.num_channels = in_channels, out_channels, tuple(num_channels)
        self.num_embeddings, self.embedding_dim = num_embeddings, embedding_dim
        self.num_res_layers, self.num_res_channels, self.num_gpus = num_res_layers, tuple(num_res_channels), num_gpus
        if latent_size is None:
            latent_size = 128 // (2 ** len(num_channels))
        self.encoder = MonaiEncoder(in_channels, embedding_dim, num_channels, num_res_layers, num_res_channels,
                                    latent_size * (2 ** len(num_channels)), downsample_parameters, dropout)
        self.decoder = MonaiDecoder(embedding_dim, out_channels, num_channels, num_res_layers, num_res_channels, latent_size,
                                    upsample_parameters, dropout, output_act, kernel_resize)
        self.quantizer = VectorQuantizer(num_embeddings, embedding_dim, layout="DK")

    def load_weights(self, path):
        _load_first_stage(self, path)


def _load_first_stage(model, path):
    """.npz of canonical names (``encoder.*``, ``decoder.*``, ``quantizer.embeddings``), or the prefix of a TensorFlow
    checkpoint of the reference's first-stage trainer (``vqvae_trainer.load_weights(ckpt)``, dm3d.py:408-414), which restores
    encoder, quantizer and decoder.  In the object graph encoder / decoder are subclassed models that hold ``self.blocks`` (a
    Sequential, or a list in vqgan_attn_cp), so their variables sit under ``<part>/blocks/...`` in layer order, and the codebook
    under ``quantizer/embeddings``.  A file without encoder tensors still loads (sampling + decode need none), but the
    encoder then refuses to run instead of encoding with random weights."""
    import os as _os
    has_enc = hasattr(model.encoder, "set_weights")
    if not str(path).endswith(".npz") and _os.path.exists(str(path) + ".index"):
        from . import tf_checkpoint as T
        variables = T.read_checkpoint(str(path))
        model.decoder.set_weights(T.assign_by_creation_order(model.decoder.spec, T.block_layer_variables(variables, "decoder/blocks")))
        if has_enc:
            enc_groups = T.block_layer_variables(variables, "encoder/blocks")
            if enc_groups:
                model.encoder.set_weights(T.assign_by_creation_order(model.encoder.spec, enc_groups))
                model.encoder.weights_missing = None
            else:
                model.encoder.weights_missing = str(path)
        emb = [v for k, v in variables.items() if k.startswith("quantizer/embeddings") and k.endswith("VARIABLE_VALUE")]
        if emb:
            model.quantizer.set_embeddings(emb[0])
        return
    p = Wt.load_npz(path)
    model.decoder.set_weights({k[len("decoder."):]: v for k, v in p.items() if k.startswith("decoder.")})
    if has_enc:
        enc = {k[len("encoder."):]: v for k, v in p.items() if k.startswith("encoder.")}
        if enc:
            model.encoder.set_weights(enc)
            model.encoder.weights_missing = None
        else:
            model.encoder.weights_missing = str(path)
    model.quantizer.set_embeddings(p["quantizer.embeddings"])


class VQGAN:
    """The VQGAN constructor surface for the path.  ``variant`` selects the reference module:
        'attn_cp' networks/vqgan_attn_cp.VQGAN (default; 32^3 <-> 128^3 with a 3-entry channel list, codebook (K,D))
        'vqgan'   networks/vqgan.VQGAN (codebook (D,K))   'gnorm' networks/vqgan_gnorm.VQGAN   'stride' networks/vqgan_stride.VQGAN
    The non-attn_cp decoders carry per-voxel PReLU alphas: ``latent_size`` fixes their resolution (Keras infers it from the
    128^3 input)."""

    def __init__(self, in_channels=1, out_channels=1, num_channels=(32, 64, 128), num_res_layers=2, num_res_channels=None,
                 num_embeddings=1024, embedding_dim=256, variant="attn_cp", latent_size=None, output_act=None, **_training_only):
        self.num_embeddings, self.embedding_dim, self.variant = num_embeddings, embedding_dim, variant
        self.encoder = _NoEncoder()
        if variant == "attn_cp":
            self.decoder = AttnCpDecoder(embedding_dim, out_channels, num_channels)
        else:
            if latent_size is None:
                latent_size = 128 // (2 ** len(num_channels))
            self.decoder = VqganFamilyDecoder(variant, embedding_dim, out_channels, num_channels, num_res_layers,
                                              num_res_channels or num_channels, latent_size, output_act)
        self.quantizer = VectorQuantizer(num_embeddings, embedding_dim, layout="DK" if variant == "vqgan" else "KD")

    def load_weights(self, path):
        _load_first_stage(self, path)
