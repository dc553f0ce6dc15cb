"""3D latent U-Net on the sm_100a kernels: the host-side mirror of ``build_model``.

    unconditional  reference networks/dm3d.py:294-376
    conditional    reference networks/conditional_dm3d.py:324-415

``build_model(img_size, img_channels, widths, has_attention, ...)`` keeps the reference's signature and
returns a ``UNet``: parameters in the reference's Keras layouts under canonical names (weights.py),
and -- once ``compile(batch, timesteps)`` is called -- a native step program of fixed-buffer kernel
launches (conv plans, fused norm+act passes, attention) that evaluates eps_hat = network([x, t(, ctx)]).

What is hoisted out of the per-step path (SURVEY K12/K9): the time-embedding MLP and every
ResidualBlock's Dense(swish(temb)) depend only on t -> tables over all T, read by the conv epilogue
through a device-side timestep; ContextMLP + key(ctx)/value(ctx) depend only on the class ids ->
computed once per generate() call.
"""
from __future__ import annotations

import math
import os
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib as L
from . import ops
from .program import Program
from . import weights as Wt


def build_model(img_size, img_channels, widths, has_attention, has_cross_attention=None, num_res_blocks=2,
                norm_groups=8, interpolation="nearest", activation_fn="swish", context_dim=None,
                first_conv_channels=None, conditional=None):
    """Same call surface as the reference's ``build_model``.  ``conditional`` defaults to the reference file
    it mirrors: dm3d.build_model (context_dim=None) is unconditional with first_conv_channels=64;
    conditional_dm3d.build_model (context_dim=1) is conditional with first_conv_channels=32.
    ``norm_groups``, ``has_cross_attention``, ``interpolation`` are accepted and unused, as in the reference."""
    if has_cross_attention and not context_dim:
        raise ValueError("Context dim can not be None if has_cross_attention is not None")
    if conditional is None:
        conditional = context_dim is not None
    if first_conv_channels is None:
        first_conv_channels = 32 if conditional else 64
    cfg = SimpleNamespace(img_size=img_size, img_channels=img_channels, widths=list(widths),
                          has_attention=list(has_attention), num_res_blocks=num_res_blocks,
                          first_conv_channels=first_conv_channels, conditional=bool(conditional),
                          context_dim=context_dim if context_dim else 1)
    return UNet(cfg)


def _walk(cfg):
    """The layer-construction order of build_model as a flat list of block records."""
    F, W, R = cfg.first_conv_channels, cfg.widths, cfg.num_res_blocks
    blocks = [dict(kind="in", name="in", cin=cfg.img_channels, cout=F, s=cfg.img_size)]
    c, s = F, cfg.img_size
    skips = [c]
    for i, w in enumerate(W):
        for j in range(R):
            blocks.append(dict(kind="res", name=f"down.{i}.res.{j}", cin=c, cskip=0, cout=w, s=s)); c = w
            if cfg.has_attention[i]:
                blocks.append(dict(kind="attn", name=f"down.{i}.attn.{j}", c=c, s=s))
            blocks.append(dict(kind="push")); skips.append(c)
        if w != W[-1]:  # the reference compares widths by VALUE (dm3d.py:343)
            blocks.append(dict(kind="down", name=f"down.{i}.downsample", c=c, s=s)); s //= 2
            blocks.append(dict(kind="push")); skips.append(c)
    blocks.append(dict(kind="res", name="mid.res.0", cin=c, cskip=0, cout=W[-1], s=s)); c = W[-1]
    blocks.append(dict(kind="attn", name="mid.attn", c=c, s=s))
    blocks.append(dict(kind="res", name="mid.res.1", cin=c, cskip=0, cout=c, s=s))
    for i in reversed(range(len(W))):
        w = W[i]
        for j in range(R + 1):
            cs = skips.pop()
            blocks.append(dict(kind="res", name=f"up.{i}.res.{j}", cin=c, cskip=cs, cout=w, s=s, pop=True)); c = w
            if cfg.has_attention[i]:
                blocks.append(dict(kind="attn", name=f"up.{i}.attn.{j}", c=c, s=s))
        if i != 0:
            blocks.append(dict(kind="up", name=f"up.{i}.upsample", c=c, s=s)); s *= 2
    blocks.append(dict(kind="out", name="out", cin=c, cout=cfg.img_channels, s=s))
    return blocks


def param_spec(cfg):
    """[(canonical name, Keras-layout shape, initialiser)] in the reference's construction order."""
    F = cfg.first_conv_channels
    sp = []
    bn = lambda n, c: [(f"{n}.gamma", (c,), "ones"), (f"{n}.beta", (c,), "zeros"), (f"{n}.mean", (c,), "zeros"), (f"{n}.var", (c,), "ones")]  # noqa: E731
    dn = lambda n, i, o, k="vs1": [(f"{n}.kernel", (i, o), k), (f"{n}.bias", (o,), "zeros")]  # noqa: E731
    cv = lambda n, k, i, o, kk="vs1": [(f"{n}.kernel", (k, k, k, i, o), kk), (f"{n}.bias", (o,), "zeros")]  # noqa: E731
    for b in _walk(cfg):
        k, n = b["kind"], b.get("name")
        if k == "in":
            sp += cv("in", 3, b["cin"], b["cout"]) + dn("time.dense0", 4 * F, 4 * F) + dn("time.dense1", 4 * F, 4 * F)
            if cfg.conditional:
                sp += [("ctx.embedding", (cfg.context_dim + 1, 4 * F), "embed")]
        elif k == "res":
            cin, w = b["cin"] + b["cskip"], b["cout"]
            if cin != w:
                sp += cv(f"{n}.shortcut", 1, cin, w)
            sp += dn(f"{n}.temb", 4 * F, w) + bn(f"{n}.norm1", cin) + cv(f"{n}.conv1", 3, cin, w) + bn(f"{n}.norm2", w) + cv(f"{n}.conv2", 3, w, w, "vs0")
        elif k == "attn":
            c, s = b["c"], b["s"]
            if not cfg.conditional:
                sp += bn(f"{n}.norm", c) + dn(f"{n}.query", c, c) + dn(f"{n}.key", c, c) + dn(f"{n}.value", c, c) + dn(f"{n}.proj", c, c, "vs0")
            else:
                sp += dn(f"{n}.ctxmlp", 4 * F, s ** 3 * c, "glorot") + bn(f"{n}.norm", c) + cv(f"{n}.proj_in", 1, c, c, "glorot")
                for q in ("norm1", "norm2", "norm3"):
                    sp += [(f"{n}.{q}.gamma", (c,), "ones"), (f"{n}.{q}.beta", (c,), "zeros")]
                sp += dn(f"{n}.query", c, c, "glorot") + dn(f"{n}.key", c, c, "glorot") + dn(f"{n}.value", c, c, "glorot")
                sp += dn(f"{n}.mlp0", c, 4 * c, "glorot") + dn(f"{n}.mlp1", 4 * c, c, "glorot") + cv(f"{n}.proj_out", 1, c, c, "glorot")
        elif k in ("down", "up"):
            sp += cv(n, 3, b["c"], b["c"])
        elif k == "out":
            sp += bn("out.norm", b["cin"]) + cv("out.conv", 3, b["cin"], b["cout"], "vs0")
    return sp


class UNet:
    """keras.Model([image_input, time_input(, context_input)]) -> eps_hat, as a compiled kernel program."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.blocks = _walk(cfg)
        self.spec = param_spec(cfg)
        self._params = None  # {name: fp32 CPU tensor, Keras layout}; random-initialised lazily
        self.prog = None
        self.weights_version = 0   # bumped by set_weights: compiled copies held elsewhere (DiffusionModel._step) key on it
        self._per_sample = None    # lazily compiled variant for a (B,) vector of distinct timesteps
        self._training = None      # lazily compiled training-mode variant (batch-statistics BatchNorm)
        self.training = False

    @property
    def params(self):
        if self._params is None:
            self._params = Wt.init_params(self.spec, seed=0, mode="keras")
        return self._params

    # ---- weights ----------------------------------------------------------------------------
    def set_weights(self, params: dict):
        Wt.check_against_spec(params, self.spec)
        self._params = {k: torch.as_tensor(np.asarray(v) if not torch.is_tensor(v) else v).float().cpu() for k, v in params.items()}
        self.prog = None
        self._per_sample = None
        self._training = None
        self.weights_version += 1

    def load_weights(self, path, name_map=None, assume_creation_order=False):
        """``path``: a flat .npz of canonical names (tools/tf_export_npz.py writes one from a reference checkpoint), or the prefix
        of a TensorFlow checkpoint (``<path>.index`` + ``<path>.data-*``, read without TensorFlow: tf_checkpoint.py) together
        with ``name_map`` -- a TF checkpoint of the functional U-Net alone does not say which layer each
        ``layer_with_weights-<n>`` is (see tf_checkpoint.load_keras_checkpoint), so without a map it is refused."""
        import os as _os
        if not str(path).endswith(".npz") and _os.path.exists(str(path) + ".index"):
            from . import tf_checkpoint as T
            self.set_weights(T.load_keras_checkpoint(str(path), self.spec, root="network", name_map=name_map,
                                                     assume_creation_order=assume_creation_order))
        else:
            self.set_weights(Wt.load_npz(path))

    def count_params(self):
        return sum(int(np.prod(s)) for _, s, _ in self.spec)

    # ---- compilation ------------------------------------------------------------------------
    def compile(self, batch: int, timesteps: int, device=None, t_dev=None, per_sample_t=False, training=False):
        """Pack weights, precompute the t-only tables, allocate every activation buffer and record the launches.
        ``per_sample_t``: the ResidualBlock time-embedding rows come from per-sample (B, w) buffers (filled by
        ``set_timesteps`` from the hoisted tables) instead of one device-side timestep for the whole batch -- the form
        train_step calls the network in (t ~ U{0..T-1} per sample, conditional_dm3d.py:474,493).
        ``training``: the program of ``network(..., training=True)`` (conditional_dm3d.py:493), on the per-sample-t form: every
        BatchNormalization normalises with the statistics of the current batch (a statistics op writes its scale / shift on the
        device before the apply pass), so none of the folds that assume constant statistics is used -- conv1 stores
        conv + temb and norm2 is a pass of its own, proj_in reads the normalised tensor, no shadow-lane norm1 halves.  The
        moving statistics are not updated: that belongs to a step that also applies gradients."""
        L.require_gpu()
        cfg, P = self.cfg, self.params
        dev = device or torch.device("cuda", torch.cuda.current_device())
        self.device, self.batch, self.timesteps = dev, batch, timesteps
        F, B, S = cfg.first_conv_channels, batch, cfg.img_size
        pr = Program(dev)
        self.prog = pr
        self.t_dev = t_dev if t_dev is not None else torch.zeros(4, dtype=torch.int32, device=dev)   # [t, t_prev, seq idx, -]
        self.training = bool(training)
        self.per_sample_t, self._temb_rows = bool(per_sample_t) or self.training, []
        g = lambda n: P[n].to(dev).contiguous()  # noqa: E731

        # --- K12: time embedding MLP for every t, then per-ResidualBlock Dense(swish(temb)) tables (T, w)
        half = 2 * F
        freqs = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1)))
        e = torch.arange(timesteps, dtype=torch.float32)[:, None] * freqs[None, :]
        sinus = torch.cat([torch.sin(e), torch.cos(e)], dim=-1).to(dev)          # TimeEmbedding (dm3d.py:177-191)
        temb = ops.dense_f32(ops.dense_f32(sinus, g("time.dense0.kernel"), g("time.dense0.bias"), act_out="silu"),
                             g("time.dense1.kernel"), g("time.dense1.bias"))      # TimeMLP (dm3d.py:280-288)
        self.temb_table = temb

        def conv(x0, kname, cout, y=None, x1=None, k=3, stride=1, mode=L.CONV_DIRECT, act=None, bias=True, chan_bias=None,
                 residual=None, y_dtype=torch.bfloat16, transposed_store=False, dense=False, out_affine=None, note="",
                 kern=None, bias_t=None, shortcut=None):
            """``shortcut``: (x, skip, name) of a 1^3 conv folded into this conv's K loop; None (nothing launched) when the
            conv's kernel cannot carry it."""
            Bx, D, H, Wd, c0 = x0.shape
            c1 = x1.shape[-1] if x1 is not None else 0
            desc = ops.make_conv_desc(mode, Bx, (D, H, Wd), c0, c1, cout, k, stride, act, None, y_dtype,
                                      chan_bias_rows=(batch if self.per_sample_t else 1) if chan_bias is not None else 0,
                                      transposed_store=transposed_store)
            if kern is None:
                kern = P[f"{kname}.kernel"]
            if dense:  # Dense on voxels == 1^3 conv: (in,out) -> (1,1,1,in,out)
                kern = kern.reshape(1, 1, 1, *kern.shape)
            wp = ops.pack_conv_weights(desc, kern).to(dev)
            if y is None:
                od, oh, ow = ops.conv_out_shape(mode, (D, H, Wd), stride)
                y = pr.buf((Bx, cout, od * oh * ow) if transposed_store else (Bx, od, oh, ow, cout), y_dtype)
            bias_dev = None if not bias else (bias_t.to(dev).contiguous() if bias_t is not None else g(f"{kname}.bias"))
            fold = None
            if shortcut is not None:
                sx, ss, sn = shortcut
                sdesc = ops.make_conv_desc(L.CONV_DIRECT, Bx, (D, H, Wd), sx.shape[-1], ss.shape[-1] if ss is not None else 0, cout, 1)
                fold = (sx, ss, ops.fold_shortcut_weights(wp, sdesc, ops.pack_conv_weights(sdesc, P[f"{sn}.kernel"])),
                        (P[f"{kname}.bias"] + P[f"{sn}.bias"]).to(dev))   # the two biases summed once, in fp32
            return pr.conv(desc, x0, wp, y, x1=x1, bias=bias_dev, chan_bias=chan_bias,
                           t_dev=self.t_dev if (chan_bias is not None and not self.per_sample_t) else None, residual=residual,
                           out_affine=out_affine, shortcut=fold, note=note or kname)

        def bgemm(a, b, y_dtype, residual=None, note=""):
            Bx, M, K = a.shape
            N = b.shape[1]
            desc = ops.make_conv_desc(L.CONV_BATCHED_GEMM, Bx, (1, 1, M), K, 0, N, 1, 1, None, None, y_dtype)
            y = pr.buf((Bx, M, N), y_dtype)
            return pr.conv(desc, a, b, y, residual=residual, note=note)

        def bn_affine(name, x0, x1=None):
            """(scale, shift) of BatchNorm ``name`` over [x0 | x1]: folded from the moving statistics, or -- training -- written
            on the device by statistics ops, each concat half from its own tensor (the statistics are per channel)."""
            if not self.training:
                return ops.bn_fold(g(f"{name}.gamma"), g(f"{name}.beta"), g(f"{name}.mean"), g(f"{name}.var"), 1e-3)
            gam, bet = g(f"{name}.gamma"), g(f"{name}.beta")
            sc, sh = pr.buf(gam.shape, torch.float32), pr.buf(gam.shape, torch.float32)
            c0 = x0.shape[-1]
            pr.bn_stats(x0, gam[:c0], bet[:c0], sc[:c0], sh[:c0], note=f"{name}.stats")
            if x1 is not None:
                pr.bn_stats(x1, gam[c0:], bet[c0:], sc[c0:], sh[c0:], note=f"{name}.stats.skip")
            pr.hold(gam, bet)
            return sc, sh

        def bn_act(x0, name, act, x1=None, note=""):
            """BatchNorm(inference) [+ swish] of x0 (or of the concat [x0, x1]) -> (y0, y1|None): the conv that reads it takes
            the two channel segments separately.  One fused norm(+concat) pass, or the x half only when the skip half was
            normalised in the shadow of the 8^3 phase.  (Writing the normalised copies from the producers' epilogues instead
            measured slower: 5.47 vs 5.08 ms/step on cfg-2, the conv epilogues are on the critical path.)"""
            sc, sh = bn_affine(name, x0, x1)
            c0 = x0.shape[-1]
            if x1 is not None and id(x1) in self.shadow_norms:
                # the skip half was normalised with this block's parameters in the shadow of the 8^3 phase (lane 4, see below):
                # only the x half is normalised here, and the conv reads the two halves as two K segments
                if not self.shadow_joined:
                    pr.sync(4, 0)
                    self.shadow_joined = True
                hs = self.shadow_norms[id(x1)]
                assert hs["name"] == name
                y0 = pr.norm_act(x0, sc[:c0].contiguous(), sh[:c0].contiguous(), pr.buf(x0.shape), act=act, note=f"{note or name}.x")
                return y0, hs["y"]
            C = c0 + (x1.shape[-1] if x1 is not None else 0)
            y = pr.buf((*x0.shape[:-1], C))
            return pr.norm_act(x0, sc, sh, y, act=act, x1=x1, note=note or name), None

        def resblock(b, x, skip):
            n, w = b["name"], b["cout"]
            cin = b["cin"] + b["cskip"]
            res = None      # width change: the 1^3 shortcut conv, with conv2 below
            if cin == w and skip is None:
                res = x
            elif cin == w:  # concat whose width equals w: materialise it once (identity affine)
                one, zero = torch.ones(cin, device=dev), torch.zeros(cin, device=dev)
                res = pr.norm_act(x, one, zero, pr.buf((*x.shape[:-1], cin)), x1=skip, note=f"{n}.concat")
            table = ops.dense_f32(temb, g(f"{n}.temb.kernel"), g(f"{n}.temb.bias"), act_in="silu")  # (T, w)
            if self.per_sample_t:   # (B, w) rows gathered from the table per call
                rows = torch.zeros(x.shape[0], w, dtype=torch.float32, device=dev)
                self._temb_rows.append((pr.hold(table), rows))
                table = rows
            h, h1 = bn_act(x, f"{n}.norm1", "silu", x1=skip)
            if self.training:   # norm2's statistics are those of conv1's output: it is stored, then normalised
                h = conv(h, f"{n}.conv1", w, x1=h1, chan_bias=pr.hold(table))
                h, _ = bn_act(h, f"{n}.norm2", "silu")
            else:
                # conv1 + temb -> BN(norm2) -> swish (dm3d.py:237-244): conv1's output has no other reader, so norm2 and the
                # activation run in conv1's epilogue on the fp32 accumulator (one HBM pass and one bf16 rounding fewer)
                sc2, sh2 = ops.bn_fold(g(f"{n}.norm2.gamma"), g(f"{n}.norm2.beta"), g(f"{n}.norm2.mean"), g(f"{n}.norm2.var"), 1e-3)
                h = conv(h, f"{n}.conv1", w, x1=h1, chan_bias=pr.hold(table), out_affine=(sc2, sh2), act="silu", note=f"{n}.conv1+norm2")
            pr.outputs[f"{n}.norm2"] = h
            if cin != w:
                # width change: the 1^3 shortcut of [x | skip] runs as the last K segment of conv2 (halo kernel), so its output is
                # never stored and read back; where conv2's kernel cannot carry it, it is a conv of its own and conv2's residual.
                # (norm1 as a side output of the shortcut conv, written from its A tiles, measured slower than the norm pass:
                # 3.35 vs 3.15 ms/step on cfg-2 -- one-tile CTAs serialise load -> transform -> store)
                y = pr.buf(h.shape)
                if conv(h, f"{n}.conv2", w, y=y, shortcut=(x, skip, f"{n}.shortcut")) is not None:
                    return y
                res = conv(x, f"{n}.shortcut", w, x1=skip, k=1)
                return conv(h, f"{n}.conv2", w, y=y, residual=res)
            return conv(h, f"{n}.conv2", w, residual=res)

        def attention_core(q, k, vT, scale, residual, note):
            # softmax(q k^T * scale) v (+ residual) in one flash-style kernel: no (B, L, L) score tensor in HBM
            return pr.attention(q, k, vT, pr.buf(q.shape), scale, residual=residual, note=f"{note}.flash")

        def attn_block(b, x):  # AttentionBlock.call (dm3d.py:39-63)
            n, c, s = b["name"], b["c"], b["s"]
            Lq = s ** 3
            B = x.shape[0]
            nrm, _ = bn_act(x, f"{n}.norm", None)
            q = conv(nrm, f"{n}.query", c, k=1, dense=True).view(B, Lq, c)
            kk = conv(nrm, f"{n}.key", c, k=1, dense=True).view(B, Lq, c)
            vT = conv(nrm, f"{n}.value", c, k=1, dense=True, transposed_store=True)
            o = attention_core(q, kk, vT, float(c) ** -0.5, None, n).view(B, s, s, s, c)
            return conv(o, f"{n}.proj", c, k=1, dense=True, residual=nrm)   # returns BN(x) + proj (dm3d.py:63)

        self.ctx_sites = []
        self._ctx_ids = None
        sites = {}

        def ctx_site(n, c, s):
            """K_ctx / V_ctx^T buffers of one attention site for the whole batch (filled by set_context)."""
            if n not in sites:
                Lq = s ** 3
                sites[n] = dict(name=n, c=c, s=s, kc=pr.buf((batch, Lq, c)), vcT=pr.buf((batch, c, Lq)))
                self.ctx_sites.append(sites[n])
            return sites[n]["kc"], sites[n]["vcT"]

        def xattn_block(b, x):  # CrossAttentionBlock.call (conditional_dm3d.py:186-195)
            n, c, s = b["name"], b["c"], b["s"]
            Lq = s ** 3
            B = x.shape[0]
            scale = float(c) ** -0.5
            # inference BatchNorm followed by the 1^3 proj_in conv is one affine map: fold it into proj_in's kernel and bias
            # (W' = diag(a) W, b' = b + shift . W; conditional_dm3d.py:187-188) -- no normalisation pass
            if self.training:   # batch statistics: normalise, then the plain proj_in
                nrm, _ = bn_act(x, f"{n}.norm", None)
                h = conv(nrm, f"{n}.proj_in", c, k=1, act="relu")
            else:
                sc_n, sh_n = ops.bn_fold(g(f"{n}.norm.gamma"), g(f"{n}.norm.beta"), g(f"{n}.norm.mean"), g(f"{n}.norm.var"), 1e-3)
                w_in = P[f"{n}.proj_in.kernel"].reshape(c, c)
                w_fold = (sc_n.cpu()[:, None] * w_in).reshape(1, 1, 1, c, c)
                b_fold = P[f"{n}.proj_in.bias"] + sh_n.cpu() @ w_in
                h = conv(x, f"{n}.proj_in", c, k=1, act="relu", kern=w_fold, bias_t=b_fold)
            gam = [g(f"{n}.norm{i}.gamma") for i in (1, 2, 3)]
            bet = [g(f"{n}.norm{i}.beta") for i in (1, 2, 3)]
            ln = pr.layernorm(h, gam, bet, [pr.buf(h.shape) for _ in range(3)], 1e-3, note=f"{n}.ln")
            hf = h.view(B, Lq, c)
            kc, vcT = ctx_site(n, c, s)
            # The three branches all read h (conditional_dm3d.py:190-192): self-attention on the caller's stream, cross
            # attention on lane 1, the MLP on lane 2 (its second GEMM adds the cross branch), and proj_out sums the two
            # partial results inside its K loop: proj_out(t1 + xs) = [t1 | xs] . [W; W]  (two K segments, no add pass).
            pr.sync(0, 1)
            pr.sync(0, 2)
            pr.sync(0, 3)
            # query(LN1(h)) and key(LN1(h)) read the same tensor: one Dense with the kernels side by side, [q | k] = x [Wq | Wk];
            # the attention kernel reads q and k as column blocks (row stride 2C) of its output
            wqk = torch.cat([P[f"{n}.query.kernel"], P[f"{n}.key.kernel"]], dim=1)
            bqk = torch.cat([P[f"{n}.query.bias"], P[f"{n}.key.bias"]])
            qk = conv(ln[0], f"{n}.query+key", 2 * c, k=1, dense=True, kern=wqk, bias_t=bqk).view(B, Lq, 2 * c)
            q1, k1 = qk[..., :c], qk[..., c:]
            pr.set_lane(3)
            v1T = conv(ln[0], f"{n}.value", c, k=1, dense=True, transposed_store=True)
            pr.set_lane(0)
            pr.sync(3, 0)
            t1 = attention_core(q1, k1, v1T, scale, hf, f"{n}.self")
            pr.set_lane(1)
            q2 = conv(ln[1], f"{n}.query", c, k=1, dense=True).view(B, Lq, c)
            c2 = attention_core(q2, kc, vcT, scale, None, f"{n}.cross")
            pr.set_lane(2)
            m = conv(ln[2], f"{n}.mlp0", 4 * c, k=1, dense=True, act="relu")
            pr.sync(1, 2)
            xs = conv(m, f"{n}.mlp1", c, k=1, dense=True, residual=c2.view(B, s, s, s, c))
            pr.set_lane(0)
            pr.sync(2, 0)
            w2 = torch.cat([P[f"{n}.proj_out.kernel"]] * 2, dim=3)
            return conv(t1.view(B, s, s, s, c), f"{n}.proj_out", c, x1=xs, k=1, act="relu", residual=x, kern=w2)

        self.x_in = pr.buf((B, S, S, S, cfg.img_channels))
        self.eps = pr.buf((B, S, S, S, cfg.img_channels), torch.float32)
        # Shadow work: the 8^3 phase of the step (a third of its time) runs kernels of 32-128 CTAs that leave most of the GPU
        # idle, and the skip tensors of the 32^3 / 16^3 levels are complete by then.  Their halves of the up-path norm1 passes
        # (BN + swish with the CONSUMER block's parameters, dm3d.py:235-236) are therefore run on lane 4 while the 8^3 phase
        # executes on the other lanes, and the up-path passes shrink to the x half.
        self.shadow_norms, self.shadow_joined = {}, False
        use_shadow = len(cfg.widths) >= 2 and not self.training   # training: the norm1 halves wait for their statistics on lane 0
        consumer, stack = {}, []          # push index -> the up-path ResidualBlock that pops it
        npush = 0
        for b in self.blocks:
            if b["kind"] in ("in", "push"):
                stack.append(npush); npush += 1
            elif b["kind"] == "res" and b.get("pop"):
                consumer[stack.pop()] = b
        deepest = min(b["s"] for b in self.blocks if b["kind"] == "res")
        shadow_done = not use_shadow

        def shadow_pass(skips, ids):
            pr.sync(0, 4)
            pr.set_lane(4)
            for t, i in zip(skips, ids):
                cb = consumer.get(i)
                if cb is None or cb["s"] == deepest or cb["cin"] + cb["cskip"] == cb["cout"]:
                    continue
                nm = f"{cb['name']}.norm1"
                sc, sh = ops.bn_fold(g(f"{nm}.gamma"), g(f"{nm}.beta"), g(f"{nm}.mean"), g(f"{nm}.var"), 1e-3)
                c0 = cb["cin"]
                y = pr.norm_act(t, sc[c0:].contiguous(), sh[c0:].contiguous(), pr.buf(t.shape), act="silu", note=f"{nm}.skip")
                self.shadow_norms[id(t)] = dict(name=nm, y=y)
            pr.set_lane(0)

        x, skips, ids = None, [], []
        next_id = 1   # push index 0 is the input conv's output
        for b in self.blocks:
            k = b["kind"]
            if not shadow_done and k == "res" and b["s"] == deepest:
                shadow_pass(skips, ids)
                shadow_done = True
            if k == "in":
                x = conv(self.x_in, "in", b["cout"])
                skips.append(x); ids.append(0)
            elif k == "res":
                skip = None
                if b.get("pop"):
                    ids.pop()
                    skip = skips.pop()
                x = resblock(b, x, skip)
            elif k == "attn":
                x = xattn_block(b, x) if cfg.conditional else attn_block(b, x)
            elif k == "push":
                skips.append(x); ids.append(next_id); next_id += 1
            elif k == "down":
                x = conv(x, b["name"], b["c"], stride=2)
            elif k == "up":
                x = conv(x, b["name"], b["c"], mode=L.CONV_PARITY)
            elif k == "out":
                h, _ = bn_act(x, "out.norm", "silu")
                conv(h, "out.conv", b["cout"], y=self.eps, y_dtype=torch.float32)
        torch.cuda.synchronize(dev)
        return self

    # ---- per-generate() context (conditional): ContextMLP + key(ctx) / value(ctx) --------------------------
    def set_context(self, ctx_ids):
        """ctx_ids: (B,) int class ids (0 healthy / 1 BraTS, dataset_utils.py:143,160)."""
        if not self.cfg.conditional:
            return
        P, dev, B = self.params, self.device, self.batch
        ids = torch.as_tensor(ctx_ids).long().reshape(-1).cpu()
        if ids.numel() == 1:
            ids = ids.expand(B)  # the reference feeds a batch-1 context (conditional_dm3d.py:552)
        assert ids.numel() == B
        if getattr(self, "_ctx_ids", None) is not None and torch.equal(self._ctx_ids, ids):
            return  # K_ctx / V_ctx^T of these class ids are already in the sites' buffers
        cemb = P["ctx.embedding"][ids].to(dev).contiguous()          # Embedding (conditional_dm3d.py:358)
        for site in self.ctx_sites:
            n, c, s = site["name"], site["c"], site["s"]
            if "dev" not in site:   # device copies of the site's weights + the two projection plans, built once
                ctxbuf = torch.empty(B, s, s, s, c, dtype=L.ACT_DTYPE, device=dev)
                plans = []
                for wname, out, tr in (("key", site["kc"], False), ("value", site["vcT"], True)):
                    desc = ops.make_conv_desc(L.CONV_DIRECT, B, (s, s, s), c, 0, c, 1, 1, transposed_store=tr)
                    wp = ops.pack_conv_weights(desc, P[f"{n}.{wname}.kernel"].reshape(1, 1, 1, c, c)).to(dev)
                    plans.append(ops.ConvPlan(desc, ctxbuf, wp, out, bias=P[f"{n}.{wname}.bias"].to(dev)))
                site["dev"] = dict(w=P[f"{n}.ctxmlp.kernel"].to(dev), b=P[f"{n}.ctxmlp.bias"].to(dev), ctx=ctxbuf, plans=plans)
            d = site["dev"]
            ctx = ops.dense_f32(cemb, d["w"], d["b"], act_out="silu")     # ContextMLP (conditional_dm3d.py:310-318)
            d["ctx"].copy_(ops.cast(ctx, L.ACT_DTYPE).view(B, s, s, s, c))
            for plan in d["plans"]:
                plan.run()
        torch.cuda.synchronize(dev)
        self._ctx_ids = ids.clone()

    # ---- call ---------------------------------------------------------------------------------------------
    def forward_inplace(self):
        """eps[...] = network(x_in, t_dev[0]) on the pre-bound buffers."""
        self.prog.run()
        return self.eps

    def set_timesteps(self, t):
        """Per-sample-t programs: gather the (B, w) time-embedding rows of ``t`` (B,) from the hoisted tables."""
        tidx = torch.as_tensor(t).reshape(-1).to(torch.int32).to(self.device)
        for table, rows in self._temb_rows:
            L.check(L.lib().b200dm_gather_rows_f32(L.ptr(table), table.shape[0], L.ptr(tidx), L.ptr(rows), rows.shape[0],
                                                  rows.shape[1], L.stream()))

    def training_program(self):
        """The training-mode compiled copy (``compile(..., training=True)``) of this compiled network, built on first use: same
        weights, own activation buffers; ``self`` and its inference program are untouched by it."""
        if self.training:
            return self
        if self._training is None:
            import copy
            self._training = copy.copy(self).compile(self.batch, self.timesteps, self.device, training=True)
        return self._training

    def __call__(self, inputs, training=False):
        """network([x (B,S,S,S,C) fp32|bf16, t (B,) int (, ctx (B,)|(B,1,1) int)], training=False) -> eps_hat fp32 (new tensor).
        ``training=True`` (train_step's call, conditional_dm3d.py:493): every BatchNormalization uses the statistics of this
        batch, so a sample's eps_hat depends on the others; the moving statistics are NOT updated (that side effect belongs to a
        step that also applies gradients).  ``training=False`` runs the inference program, unchanged by training calls."""
        x, t = inputs[0], inputs[1]
        if self.prog is None or self.batch != x.shape[0]:
            raise L.B200dmError("UNet: call compile(batch, timesteps) first (batch must match)")
        tvec = torch.as_tensor(t).reshape(-1).to(torch.int64).cpu()
        if tvec.numel() == 1:
            tvec = tvec.expand(x.shape[0])
        if tvec.numel() != x.shape[0] or int(tvec.min()) < 0 or int(tvec.max()) >= self.timesteps:
            raise L.B200dmError(f"UNet: t must hold {x.shape[0]} timesteps in [0, {self.timesteps})")
        if bool(training) != self.training:
            if not training:
                raise L.B200dmError("UNet: this is the training-mode program; call the network it was built from")
            return self.training_program()(inputs, training=True)
        tv = int(tvec[0])
        if not bool((tvec == tv).all()) and not self.per_sample_t:
            # distinct timesteps per sample (train_step's call, conditional_dm3d.py:493): a second compiled program whose conv
            # epilogues read per-sample (B, w) time-embedding rows; same packed weights, own activation buffers
            if self._per_sample is None:
                import copy
                self._per_sample = copy.copy(self).compile(self.batch, self.timesteps, self.device, per_sample_t=True)
            return self._per_sample(inputs)
        if len(inputs) > 2 and self.cfg.conditional:
            self.set_context(torch.as_tensor(inputs[2]).reshape(-1))
        if self.per_sample_t:
            self.set_timesteps(tvec)
        self.t_dev.copy_(torch.tensor([tv, tv - 1, 0, 0], dtype=torch.int32))
        x = x.to(self.device)
        self.x_in.copy_(x if x.dtype == L.ACT_DTYPE else ops.cast(x.contiguous().float(), L.ACT_DTYPE))
        return self.forward_inplace().clone()
