"""Latent diffusion wrapper: the host-side mirror of the reference's ``DiffusionModel``.

    unconditional  networks/dm3d.py:379-545          (generate :510-532, sample :477-508, test :534-545)
    conditional    networks/conditional_dm3d.py:418-594 (generate :550-575, test :577-593)

Same constructor ``DiffusionModel(latent_size, num_embed, latent_channels, vqvae_load_ckpt, args)`` (``args`` carries
timesteps / num_gpus / kernel_resize / bs), same attributes (.timesteps .b .network .encoder .quantizer .decoder
.vqvae_trainer) and the same ``sample(x_t, pred_noise, t, shape) -> (mean, var)`` and
``generate(shape, last_step[, context_value]) -> latents`` contracts.  Build additions (explicit extensions,
SURVEY 8b): ``x_T=``, ``noise=`` (inject), ``seed=``, ``sample_id0=`` (multi-GPU sharding), ``sampler="ddim"``,
``steps=``, per-sample ``context=`` ids, ``decode(latents, quantize=False)`` and ``train_loss`` (the forward half of
train_step and its loss, without gradients).

The reverse loop is one captured CUDA graph per step: U-Net program + fused posterior update + a device-side
timestep decrement, replayed T times with zero host work in between.  Samples are independent (BatchNorm in inference
mode, per-sample attention), so the batch can be split into ``chains`` sub-batches whose kernel chains are captured on
parallel graph branches (B200DM_CHAINS; default 1 -- measured no gain on B200, see _num_chains).
"""
from __future__ import annotations

import copy
import ctypes
import os

import numpy as np
import torch

from . import _lib as L
from . import ops
from .first_stage import VQVAE
from .program import Program
from .unet import build_model


class Betas(ops.ScheduleTables):
    """reference ``Betas`` (dm3d.py:194-214): attribute access to the fp32 tables."""

    def __getattr__(self, k):
        host = self.__dict__.get("host", {})
        if k in host:
            return host[k]
        raise AttributeError(k)


class DiffusionModel:
    conditional = False
    first_conv_channels = 64

    def __init__(self, latent_size, num_embed, latent_channels, vqvae_load_ckpt, args, first_stage=None):
        self.timesteps = args.timesteps
        self.b = Betas(args.timesteps)
        self.lc = latent_channels
        self.latent_size = latent_size
        self.num_gpus, self.global_bs = getattr(args, "num_gpus", 1), getattr(args, "bs", 1)
        # The unconditional file hard-codes K=1024, D=256 (dm3d.py:405-406); the conditional one uses the arguments
        # (conditional_dm3d.py:444-445).  ``first_stage`` lets a caller plug any object with .encoder/.quantizer/.decoder.
        if first_stage is None:
            K, D = (num_embed, latent_channels) if self.conditional else (1024, 256)
            first_stage = VQVAE(in_channels=1, out_channels=1, num_channels=(32, 64, 128, 256),
                                num_res_channels=(32, 64, 128, 256), num_res_layers=5,
                                downsample_parameters=((2, 4, 1, "same"),) * 4, upsample_parameters=((2, 4, 1, "same", 0),) * 4,
                                num_embeddings=K, embedding_dim=D, dropout=None,
                                num_gpus=self.num_gpus, kernel_resize=getattr(args, "kernel_resize", False),
                                latent_size=latent_size)
        self.vqvae_trainer = first_stage
        self.vqvae_load_ckpt = vqvae_load_ckpt
        if vqvae_load_ckpt is not None:
            print("Loading VQVAE weights")
            self.vqvae_trainer.load_weights(vqvae_load_ckpt)
        self.encoder, self.quantizer, self.decoder = first_stage.encoder, first_stage.quantizer, first_stage.decoder
        self.network = build_model(latent_size, latent_channels, widths=[64, 128, 256],
                                   has_attention=[False, False, True, True],
                                   context_dim=1 if self.conditional else None,
                                   first_conv_channels=self.first_conv_channels, conditional=self.conditional)
        self._step = None
        self._train = None

    # ------------------------------------------------------------------ reference API
    def load_weights(self, path):
        self.network.load_weights(path)
        self._step = None
        self._train = None

    def sample(self, x_t, pred_noise, curr_time_step, shape=None):
        """-> (posterior_mean, variance); the reference returns the variance under the name log-variance
        (dm3d.py:506-508).  Standalone diagnostic form with the reference's fp32 op order; inside generate() the same
        arithmetic runs fused with the clip and the noise add in the update kernel (csrc/update.cu)."""
        t = int(torch.as_tensor(curr_time_step).reshape(-1)[0])
        h = self.b.host
        f = lambda n: torch.tensor(h[n][t], dtype=torch.float32, device=x_t.device)  # noqa: E731
        x_0 = (x_t - f("sqrt_one_minus_alpha_bar") * pred_noise) / f("sqrt_alpha_bar")
        mean = (f("beta") * f("sqrt_alpha_bar_prev") / (1 - f("alpha_bar"))) * x_0 + \
               ((1 - f("alpha_bar_prev")) * f("sqrt_alpha") / (1 - f("alpha_bar"))) * x_t
        var = (1 - f("alpha_bar_prev")) * f("beta") / (1 - f("alpha_bar"))
        return mean, var.reshape(1, 1, 1, 1, 1).expand(x_t.shape[0], 1, 1, 1, 1)

    # ------------------------------------------------------------------ compiled step
    @staticmethod
    def _num_chains(batch):
        # default 1: measured on B200 (cfg-2, B=8) 1 chain 4.98 ms/step, 2 chains 5.22, 4 chains 5.31 -- the persistent
        # 148-CTA conv kernels of one chain leave no SMs for the other chain's small kernels, and smaller sub-batches
        # make the 8^3-level GEMM grids even thinner
        want = int(L.tuning_env("B200DM_CHAINS", "1"))
        c = max(1, min(want, batch))
        while batch % c:
            c -= 1
        return c

    def _compile(self, batch, sampler, inject_noise, seed, sample_id0, fuse_update=False):
        # the compiled copies hold PACKED weights: key on the network's weights version so that network.set_weights /
        # network.load_weights (INTEGRATION.md) is never followed by sampling with the old weights
        key = (batch, sampler, inject_noise, self._num_chains(batch), self.network.weights_version, bool(fuse_update))
        if self._step is not None and self._step["key"] == key:
            return self._step   # seed / sample base are device-resident (t_dev[4..7]): the captured graph serves every call
        L.require_gpu()
        dev = torch.device("cuda", torch.cuda.current_device())
        self.b.to(dev)
        t_dev = torch.zeros(8, dtype=torch.int32, device=dev)        # [t, t_prev, sequence index, -, seed lo, hi, sample base lo, hi]
        t_seq = torch.full((self.timesteps + 2,), -1, dtype=torch.int32, device=dev)   # the call's timestep sequence, -1 terminated
        chains = key[3]
        cb = batch // chains
        # one compiled program per chain: shallow copies of self.network (weights shared on the host, buffers per chain)
        nets = [copy.copy(self.network).compile(cb, self.timesteps, dev, t_dev=t_dev) for _ in range(chains)]
        S, Cl = self.latent_size, self.lc
        x = torch.zeros(batch, S, S, S, Cl, dtype=torch.float32, device=dev)
        noise = torch.zeros_like(x) if inject_noise else None
        descs = [ops.make_update_desc(self.b, x[0].numel(), cb, 0, -1, 1 if sampler == "ddim" else 0, 0,
                                      c * cb, L.F32, t_dev=t_dev, seed_on_device=True) for c in range(chains)]
        # Fused update: the output conv's epilogue turns its eps tile straight into x_{t-1} (+ the 16-bit copy that is the next
        # step's network input) -- no fp32 eps round trip through HBM, no update launch.  Same arithmetic and noise stream as
        # the update kernel (bit-identical latents); needs the Philox path (no injected noise) and an output conv on the
        # CTA-pair fp32 kernel (C_lat % 128 == 0, planes >= 8 x 16), else the two-kernel form stays.
        fused = False
        if fuse_update and not inject_noise:
            oks = []
            for c, net in enumerate(nets):
                plan = net.prog.producers.get(net.eps.data_ptr())
                xs = x[c * cb:(c + 1) * cb]
                oks.append(plan is not None and plan.set_fused_update(descs[c], xs, xs, net.x_in))
            fused = all(oks)
            assert fused or not any(oks), "fused update: the chains' output convs differ"
        self._step = dict(key=key, nets=nets, net=nets[0], x=x, noise=noise, descs=descs, t_dev=t_dev, t_seq=t_seq, graph=None, dev=dev,
                          chains=chains, chain_batch=cb, streams=None, fused=fused)
        return self._step

    def _run_chain(self, st, c):
        """U-Net forward of chain c -> fused update of its samples (x in place, bf16 copy into the U-Net input)."""
        cb, net = st["chain_batch"], st["nets"][c]
        net.prog.run()
        if st["fused"]:   # the output conv has already written x_{t-1} and the next network input
            return
        xs = st["x"][c * cb:(c + 1) * cb]
        nz = st["noise"][c * cb:(c + 1) * cb] if st["noise"] is not None else None
        L.check(L.lib().b200dm_ddpm_update(ctypes.byref(st["descs"][c]), L.ptr(xs), L.ptr(net.eps), L.ptr(nz), L.ptr(xs),
                                           L.ptr(net.x_in), L.stream()))

    def _run_step_eager(self, st, parallel=False):
        """Every chain's forward + update, then t_dev moves to the next entry of the device-resident timestep sequence.
        ``parallel``: fork the chains onto side streams (inside a graph capture this records parallel branches)."""
        if parallel and st["chains"] > 1:
            if st["streams"] is None:
                st["streams"] = [torch.cuda.Stream() for _ in range(st["chains"] - 1)]
            main = torch.cuda.current_stream()
            for c, s in enumerate(st["streams"], start=1):
                s.wait_stream(main)
                with torch.cuda.stream(s):
                    self._run_chain(st, c)
            self._run_chain(st, 0)
            for s in st["streams"]:
                main.wait_stream(s)
        else:
            for c in range(st["chains"]):
                self._run_chain(st, c)
        L.check(L.lib().b200dm_step_advance_seq(L.ptr(st["t_dev"]), L.ptr(st["t_seq"]), L.stream()))

    def _capture(self, st):
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._run_step_eager(st, parallel=True)  # warm-up (sets kernel attributes outside capture)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            self._run_step_eager(st, parallel=True)
        st["graph"] = g
        return g

    def generate(self, shape=(1, 16, 16, 16, 16), last_step=0, context_value=None, *, x_T=None, noise=None, seed=None,
                 sample_id0=0, sampler="ddpm", steps=None, context=None, use_graph=True, on_step=None, timestep_seq=None,
                 fuse_update=None):
        """Reverse diffusion from t=T-1 down to ``last_step`` (dm3d.py:510-532).  ``noise``: callable i -> tensor or
        dict/sequence indexed by timestep, injected instead of the Philox stream (parity tests).  ``seed=None`` draws a fresh
        seed per call (the reference draws fresh tf.random.normal noise on every call); it is kept in ``self.last_seed``.
        ``sampler="ddim"`` with ``steps=n`` (or an explicit descending ``timestep_seq``) walks a sub-sequence of the schedule.
        ``fuse_update`` (default: on when possible) runs the update inside the output conv's epilogue (see _compile).
        The timestep sequence lives in device memory and the captured step graph indexes it, so every sequence -- DDPM ranges,
        strided or non-uniform DDIM -- replays the same graph with no host work between steps.  Returns fp32 latents."""
        shape = tuple(shape)
        B = shape[0]
        assert shape[1] == self.latent_size and shape[-1] == self.lc, "shape must match the compiled latent geometry"
        if seed is None:
            seed = int.from_bytes(os.urandom(7), "little")
        self.last_seed = seed
        if fuse_update is None:   # default: on whenever nothing needs eps_hat in HBM
            fuse_update = noise is None and on_step is None
        assert not (fuse_update and (noise is not None or on_step is not None)), "fuse_update: no injected noise / eps callback"
        st = self._compile(B, sampler, noise is not None, seed, sample_id0, fuse_update)
        dev, nets, cb = st["dev"], st["nets"], st["chain_batch"]
        if self.conditional:
            ctx = context if context is not None else (0 if context_value is None else context_value)
            ctx = torch.as_tensor(ctx).reshape(-1)
            if ctx.numel() == 1:
                ctx = ctx.expand(B)  # the reference feeds a batch-1 context (conditional_dm3d.py:552)
            for c, net in enumerate(nets):
                net.set_context(ctx[c * cb:(c + 1) * cb])
        T = self.timesteps
        if timestep_seq is not None:
            seq = [int(v) for v in timestep_seq]
            assert all(0 <= v < T for v in seq) and all(a > b for a, b in zip(seq, seq[1:])), "timestep_seq: descending values in [0, T)"
        elif sampler == "ddim":
            n = steps or T
            seq = sorted({int(round(v)) for v in np.linspace(last_step, T - 1, n)}, reverse=True)
        else:
            seq = list(range(T - 1, last_step - 1, -1))
        if not seq:
            raise ValueError("generate: empty timestep sequence")
        # one small H2D per call: the whole sequence (+ the -1 terminators) and the walker's start state
        st["t_seq"].copy_(torch.tensor(seq + [-1] * (T + 2 - len(seq)), dtype=torch.int32), non_blocking=True)
        i32 = lambda v: v - (1 << 32) if v >= (1 << 31) else v  # noqa: E731
        start = torch.tensor([seq[0], seq[1] if len(seq) > 1 else -1, 0, 0, i32(seed & 0xffffffff), i32((seed >> 32) & 0xffffffff),
                              i32(sample_id0 & 0xffffffff), i32((sample_id0 >> 32) & 0xffffffff)], dtype=torch.int32)
        if x_T is None:  # samples = tf.random.normal(shape) (dm3d.py:513): Philox stream 1
            x0, xb = ops.philox_normal(shape, seed, sample_id0, 0, 1, want_bf16=True)
        else:
            x0 = x_T.to(dev, torch.float32, non_blocking=True).contiguous()
            xb = ops.cast(x0, L.ACT_DTYPE)

        def load_state():
            st["x"].copy_(x0)
            for c, net in enumerate(nets):
                net.x_in.copy_(xb[c * cb:(c + 1) * cb])
            st["t_dev"].copy_(start, non_blocking=True)

        load_state()
        if use_graph and noise is None and on_step is None:
            if st["graph"] is None:
                self._capture(st)   # runs one warm-up step + records one: restore the state afterwards
                load_state()
            for _ in seq:
                st["graph"].replay()
        else:
            for i in seq:
                if noise is not None and i > 0:
                    z = noise(i) if callable(noise) else noise[i]
                    st["noise"].copy_(z.to(dev, torch.float32))
                self._run_step_eager(st)
                if on_step is not None:
                    on_step(i, st["x"], torch.cat([net.eps for net in nets], 0))
        return st["x"].clone()

    def encode(self, images):
        """``latents, _ = self.quantizer(self.encoder(images))`` -- the first line of the reference's train_step
        (dm3d.py / conditional_dm3d.py:478): volumes (B,S,S,S,1) -> quantised latents (B,s,s,s,D) fp32 on the device."""
        latents, _ = self.quantizer(self.encoder(images))
        return latents

    def _t_dev(self, t, B):
        t = torch.as_tensor(t).reshape(-1).long().cpu()
        if t.numel() == 1:
            t = t.expand(B)
        if t.numel() != B or int(t.min()) < 0 or int(t.max()) >= self.timesteps:
            raise ValueError(f"t must hold {B} timesteps in [0, {self.timesteps})")
        return t, t.to(torch.int32).cuda()

    def q_sample(self, latents, t, noise):
        """Forward diffusion of train_step (conditional_dm3d.py:484-490): sqrt(abar_t) * latents + sqrt(1 - abar_t) * noise,
        t (B,) int, in the reference's fp32 op order -> fp32 x_t on the device (the q-sample kernel of train_loss)."""
        L.require_gpu()
        self.b.to(torch.device("cuda", torch.cuda.current_device()))
        z = latents.cuda().float().contiguous()
        _, t_dev = self._t_dev(t, z.shape[0])
        return ops.q_sample(self.b, z, t_dev, noise=noise.to(z.device, torch.float32).contiguous(), want_f32=True)[1]

    @staticmethod
    def draw_timesteps(seed, batch, timesteps):
        """t ~ U{0..T-1} per sample (conditional_dm3d.py:474) from a host generator seeded with ``seed``: reproducible."""
        g = torch.Generator().manual_seed(int(seed))
        return torch.randint(0, timesteps, (batch,), generator=g, dtype=torch.int64)

    def loss_divisor(self):
        """global_bs * lc^4: train_step divides the summed MSE by this literal (conditional_dm3d.py:496-499, SURVEY 3.5)."""
        return float(self.global_bs) * float(self.lc) ** 4

    def train_loss(self, images=None, *, latents=None, context=None, t=None, noise=None, seed=None):
        """The loss train_step computes (conditional_dm3d.py:471-499), without the gradient step: ``latents`` (or the frozen
        ``encode(images)``) -> t ~ U{0..T-1} per sample from a host generator seeded with ``seed`` (unless ``t`` is given) ->
        x_t = q_sample(latents, t, noise) with the noise from Philox stream 2 of ``seed`` (unless ``noise`` is injected) ->
        eps_hat = network([x_t, t, ctx], training=True) (batch-statistics BatchNorm, moving statistics not updated) ->
        MSE(reduction=SUM)(noise, eps_hat) / (global_bs * lc^4).  BatchNorm statistics are those of this process's batch, as on a
        MirroredStrategy replica; ``global_bs`` is ``args.bs``.  ``seed=None`` draws a fresh seed (kept in ``last_seed``; the t
        used in ``last_t``).  Returns the loss as a 0-d fp32 tensor on the device."""
        if latents is None:
            if images is None:
                raise ValueError("train_loss: give images or latents")
            latents = self.encode(images)
        L.require_gpu()
        dev = torch.device("cuda", torch.cuda.current_device())
        z = latents.to(dev, torch.float32).contiguous()
        B = z.shape[0]
        if tuple(z.shape[1:]) != (self.latent_size,) * 3 + (self.lc,):
            raise ValueError(f"train_loss: latents {tuple(z.shape)} do not match the latent geometry")
        if seed is None:
            seed = int.from_bytes(os.urandom(7), "little")
        self.last_seed = seed
        if t is None:
            t = self.draw_timesteps(seed, B, self.timesteps)
        t, t_dev = self._t_dev(t, B)
        self.last_t = t.clone()
        key = (B, self.network.weights_version)
        if self._train is None or self._train["key"] != key:
            self.b.to(dev)
            self._train = dict(key=key, net=copy.copy(self.network).compile(B, self.timesteps, dev, training=True))
        net = self._train["net"]
        if self.conditional:
            ctx = torch.as_tensor(0 if context is None else context).reshape(-1)
            net.set_context(ctx.expand(B) if ctx.numel() == 1 else ctx)
        if noise is not None:
            noise = noise.to(dev, torch.float32).contiguous()
        net.set_timesteps(t)
        ops.q_sample(self.b, z, t_dev, noise=noise, seed=seed, out16=net.x_in)
        net.forward_inplace()
        return ops.noise_loss(net.eps, self.loss_divisor(), noise=noise, seed=seed)[0]

    def decode(self, latents, quantize=False):
        """latents -> volumes through the first-stage decoder; ``quantize=True`` snaps latents to the codebook first
        (extension: the reference's test() decodes un-quantized latents, dm3d.py:541)."""
        if quantize:
            latents, _, _ = self.quantizer.quantize(latents, q_dtype=L.ACT_DTYPE)   # the decoder's input dtype: no cast pass
        return self.decoder(latents)

    def test(self, test_prefix, context=None, shape=None, out_dir="./generated_images_dm3d", **gen_kw):
        """reference test(): generate (10,16,16,16,64) latents, decode, save .npy (dm3d.py:534-545).  The literal shape
        is a default; pass ``shape`` to override (the reference's literals are mutually inconsistent, SURVEY A13).  Extra keyword
        arguments (seed=, sampler=, steps=, x_T=, noise=) go to generate()."""
        i = self.timesteps
        print(f"Generating for {i} rsteps")
        if self.vqvae_load_ckpt is not None:
            self.vqvae_trainer.load_weights(self.vqvae_load_ckpt)
        shape = shape or (10, self.latent_size, self.latent_size, self.latent_size, self.lc)
        kw = dict(context_value=context) if self.conditional and context is not None else {}
        lat = self.generate(shape, last_step=self.timesteps - i, **{**kw, **gen_kw})
        images = self.decoder(lat)
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, f"{test_prefix}-{i}rsteps.npy"), images.cpu().numpy())
        return images


class ConditionalDiffusionModel(DiffusionModel):
    """networks/conditional_dm3d.DiffusionModel: first_conv_channels=32, class-id context -> cross-attention."""
    conditional = True
    first_conv_channels = 32
