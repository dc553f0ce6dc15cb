"""GPU parity of the assembled path: U-Net forward (uncond + cond), decoders, VQ+decode, and the full
reverse chain with injected noise -- product (CUDA, through the C ABI) vs oracle (CPU).

Tolerances (stated, and why):
  * every kernel accumulates in fp32, so on IDENTICAL inputs a layer matches the oracle to ~1e-6 (tests/test_conv_gpu.py);
    test_unet_layer_trace pins that inside the assembled network: 'in' conv rel-L2 <= 1e-5 and the first ResidualBlock
    <= 1e-3 (4e-3 behind the fused conv1+norm2 epilogue, which skips one 16-bit rounding) against the oracle that rounds to the storage type at the same storage points (emu16()).
  * activations are STORED in bf16 (north_star).  A network of ~100 bf16 storage points is chaotic at the ulp level:
    one rounding flip (4e-3 of an element) perturbs 27*C downstream sums and flips more, so after ~10 layers the
    product and the emulating oracle are decorrelated at the bf16 noise floor.  The whole-network bound is therefore
    the bf16 storage error itself: eps_hat rel-L2 <= 2.5e-2 against BOTH the fp32 oracle and the emulating oracle
    (measured 1.4e-2; the two oracles differ from each other by 1.5e-2 with these stress-initialised weights).
  * chain (T steps, injected noise): latents rel-L2 <= 1e-2, max-abs <= 5e-2 against the emulating oracle
    (measured 3e-3 / 1.5e-2 at T=12: the posterior update damps eps_hat error, it does not compound it).
  * the fp16 storage build (tests/test_fp16_build_gpu.py runs this file there) has 8x smaller storage rounding: each storage-floor
    bound is tol(bf16, fp16), the fp16 value set from the error measured in that build with the margin the bf16 bound has.
"""
import types

import numpy as np
import pytest
import torch

from oracle import init as OI, ops as O, sampler as OS
from oracle.ops import Emu
from oracle.schedule import Betas as OBetas
from oracle.unet import UNet as OUNet
from oracle import first_stage as OF

pytestmark = pytest.mark.gpu


def tol(bf16, fp16):
    """A storage-floor bound: its value in the bf16 build and in the fp16 build (8x smaller storage rounding)."""
    from b200dm import _lib
    return bf16 if _lib.precision() == "bf16" else fp16


def emu16():
    """The oracle that rounds to the build's 16-bit storage type where the CUDA path stores."""
    from b200dm import _lib
    return Emu(True, dtype=_lib.ACT_DTYPE)


def rel(a, b):
    return ((a.float().cpu() - b).norm() / (b.norm() + 1e-20)).item()


def _unet_pair(S, C_lat, cond, seed=0):
    import b200dm
    F = 32 if cond else 64
    net = b200dm.build_model(S, C_lat, [64, 128, 256], [False, False, True, True], context_dim=1 if cond else None)
    ou = OUNet(S, C_lat, [64, 128, 256], [False, False, True, True], first_conv_channels=F, conditional=cond)
    P = OI.make_params(ou.spec(), seed, "stress")
    net.set_weights(P)
    return net, ou, P


@pytest.mark.parametrize("S,C_lat,B", [(8, 8, 2), (16, 8, 1)])
def test_unet_uncond_forward(cuda, S, C_lat, B):
    net, ou, P = _unet_pair(S, C_lat, False)
    net.compile(B, 50)
    x = OI.normal((B, S, S, S, C_lat), 1)
    for t in (37, 0):
        tt = torch.full((B,), t)
        y = net([x.to(cuda), tt])
        from b200dm import _lib
        assert _lib.debug_flag() == 0
        ref_e = ou.forward(P, x, tt, emu=emu16())
        ref_x = ou.forward(P, x, tt)
        r_e, r_x = rel(y, ref_e), rel(y, ref_x)
        print(f"uncond S={S} t={t}: rel-L2 vs bf16-emulating oracle {r_e:.3e}, vs fp32 oracle {r_x:.3e}")
        assert r_e <= tol(2.5e-2, 3.2e-3), r_e
        assert r_x <= tol(2.5e-2, 3.2e-3), r_x


def test_unet_layer_trace(cuda):
    """Kernel exactness inside the assembled network, before bf16 chaos sets in."""
    S, C_lat, B = 8, 8, 2
    net, ou, P = _unet_pair(S, C_lat, False)
    net.compile(B, 50)
    x = OI.normal((B, S, S, S, C_lat), 1)
    tt = torch.full((B,), 37)
    net([x.to(cuda), tt])
    tr = {}
    ou.forward(P, x, tt, emu=Emu(True, tr, dtype=emu16().dtype))
    errs = {k: rel(v.reshape(tr[k].shape), tr[k]) for k, v in net.prog.outputs.items() if k in tr}
    print("layer trace:", {k: f"{errs[k]:.2e}" for k in ("in", "down.0.res.0.norm1", "down.0.res.0.norm2", "down.0.res.0.conv2")},
          f"max {max(errs.values()):.2e}")
    assert errs["in"] <= tol(1e-5, 5e-5), errs["in"]   # fp16: rounding flips of the stored output (~1 in 2e3 elements)
    # conv1 -> norm2 -> swish is ONE kernel (BN applied to the fp32 accumulator): the emulating oracle rounds conv1's
    # output to bf16 first, so that tensor differs by one extra bf16 rounding (<= 2^-8 per element)
    for k, bound in (("down.0.res.0.norm1", tol(1e-3, 1e-4)), ("down.0.res.0.norm2", tol(4e-3, 5e-4)),
                     ("down.0.res.0.conv2", tol(4e-3, 5e-4))):
        assert errs[k] <= bound, (k, errs[k])
    assert max(errs.values()) <= tol(2.5e-2, 3.2e-3)


def test_unet_cond_forward(cuda):
    S, C_lat, B = 8, 16, 2
    net, ou, P = _unet_pair(S, C_lat, True)
    net.compile(B, 50)
    x = OI.normal((B, S, S, S, C_lat), 1)
    ctx = torch.tensor([0, 1])
    tt = torch.full((B,), 21)
    y = net([x.to(cuda), tt, ctx])
    ref_e = ou.forward(P, x, tt, ctx=ctx, emu=emu16())
    ref_x = ou.forward(P, x, tt, ctx=ctx)
    r_e, r_x = rel(y, ref_e), rel(y, ref_x)
    print(f"cond: rel-L2 vs bf16-emulating oracle {r_e:.3e}, vs fp32 oracle {r_x:.3e}")
    assert r_e <= tol(2.5e-2, 3.2e-3) and r_x <= tol(2.5e-2, 3.2e-3)
    # context must matter and be per-sample
    y2 = net([x.to(cuda), tt, torch.tensor([1, 1])])
    assert rel(y2[1:], y[1:].cpu()) < 1e-6 and rel(y2[:1], y[:1].cpu()) > 1e-4


def test_full_chain_injected_noise(cuda):
    """T-step DDPM chain, same x_T and per-step noise on both sides (SURVEY A12)."""
    import b200dm
    S, C_lat, B, T = 8, 8, 2, 12
    args = types.SimpleNamespace(timesteps=T, num_gpus=1, kernel_resize=False, bs=B)
    dm = b200dm.DiffusionModel(S, 256, C_lat, None, args)
    ou = OUNet(S, C_lat, [64, 128, 256], [False, False, True, True], first_conv_channels=64)
    P = OI.make_params(ou.spec(), 0, "stress")
    dm.network.set_weights(P)
    shape = (B, S, S, S, C_lat)
    x_T = OI.normal(shape, 1234)
    noises = {i: OI.normal(shape, 100 + i) for i in range(1, T)}
    lat = dm.generate(shape, x_T=x_T, noise=noises)
    ob = OBetas(T)
    emu = emu16()
    ref = OS.generate(lambda x, i: ou.forward(P, x, torch.full((B,), i), emu=emu), ob, x_T, noises=noises)
    r = rel(lat, ref)
    ma = (lat.cpu() - ref).abs().max().item()
    print(f"chain T={T}: rel-L2 {r:.3e} max-abs {ma:.3e}")
    assert r <= tol(1e-2, 1.2e-3) and ma <= tol(5e-2, 6e-3), (r, ma)
    # graph path with the Philox stream == eager path with the oracle's Philox noise injected
    lat_g = dm.generate(shape, x_T=x_T, seed=77)
    from oracle import philox
    n_elem = int(np.prod(shape[1:]))
    inj = {i: torch.from_numpy(philox.normal(77, i, np.arange(B), n_elem)).reshape(shape) for i in range(1, T)}
    lat_e = dm.generate(shape, x_T=x_T, noise=inj)
    # (the two noise streams agree to ~1e-6; the chain amplifies that like any other ulp-level perturbation)
    print(f"graph + Philox vs eager + injected: rel-L2 {rel(lat_g, lat_e.cpu()):.3e}")
    assert rel(lat_g, lat_e.cpu()) <= tol(5e-3, 8e-4), rel(lat_g, lat_e.cpu())
    # sharding invariance: sample 1 generated alone with sample_id0=1 equals row 1 of the batch
    dm1 = b200dm.DiffusionModel(S, 256, C_lat, None, args)
    dm1.network.set_weights(P)
    lat_1 = dm1.generate((1,) + shape[1:], x_T=x_T[1:], seed=77, sample_id0=1)
    print(f"sample 1 alone vs in the batch: rel-L2 {rel(lat_1, lat_g[1:].cpu()):.3e}")
    assert rel(lat_1, lat_g[1:].cpu()) <= tol(5e-3, 8e-4), rel(lat_1, lat_g[1:].cpu())


def test_monai_decoder(cuda):
    import b200dm
    dec = b200dm.MonaiDecoder(64, 1, (32, 64), 2, (32, 64), 4)
    od = OF.MonaiDecoder(64, 1, (32, 64), 2, (32, 64), 4)
    P = OI.make_params(od.spec(), 5, "stress")
    dec.set_weights(P)
    z = OI.normal((2, 4, 4, 4, 64), 11)
    y = dec(z.to(cuda))
    assert tuple(y.shape) == (2, 16, 16, 16, 1) and y.dtype == torch.float32
    r_e, r_x = rel(y, od.forward(P, z, emu16())), rel(y, od.forward(P, z))
    print(f"monai decoder: rel-L2 vs emu {r_e:.3e}, vs fp32 {r_x:.3e}")
    assert r_e <= tol(8e-3, 1.2e-3) and r_x <= tol(3e-2, 4e-3)


def test_monai_encoder_and_quantize(cuda):
    """volumes -> Encoder (k4 s2 'same' convs, ResUnits, per-voxel PReLU) -> quantizer: the front half of train_step
    (conditional_dm3d.py:478: latents, _ = self.quantizer(self.encoder(images)))."""
    import b200dm
    enc = b200dm.MonaiEncoder(1, 8, (32, 64), 1, (32, 64), 16)
    oe = OF.MonaiEncoder(1, 8, (32, 64), 1, (32, 64), 16)
    P = OI.make_params(oe.spec(), 6, "stress")
    enc.set_weights(P)
    vol = OI.normal((2, 16, 16, 16, 1), 12)
    z = enc(vol.to(cuda))
    assert tuple(z.shape) == (2, 4, 4, 4, 8) and z.dtype == torch.float32
    r_e, r_x = rel(z, oe.forward(P, vol, emu16())), rel(z, oe.forward(P, vol))
    print(f"monai encoder: rel-L2 vs emu {r_e:.3e}, vs fp32 {r_x:.3e}")
    assert r_e <= tol(8e-3, 1.2e-3) and r_x <= tol(3e-2, 4e-3)
    # quantise the SAME latents on both sides: indices bit-exact (the encoder's own rounding noise is tested above)
    vq = b200dm.VectorQuantizer(64, 8, layout="DK")
    cb = OI.codebook(64, 8, "DK", seed=3)
    vq.set_embeddings(cb)
    q, idx, _ = vq.quantize(z)
    q_ref, idx_ref, _, _ = OF.quantize(z.cpu(), cb, "DK")
    assert torch.equal(idx.cpu(), idx_ref) and torch.equal(q.cpu(), q_ref)
    # train_step's forward half through the model surface: encode -> q_sample (conditional_dm3d.py:478-490)
    dm = b200dm.DiffusionModel(4, 64, 8, None, types.SimpleNamespace(timesteps=50, num_gpus=1, kernel_resize=False, bs=2))
    dm.vqvae_trainer.encoder, dm.encoder = enc, enc
    dm.vqvae_trainer.quantizer, dm.quantizer = vq, vq
    lat = dm.encode(vol.to(cuda))
    assert torch.equal(lat.cpu(), q_ref)
    t, nz = torch.tensor([3, 40]), OI.normal(tuple(lat.shape), 13)
    b = OBetas(50)
    want = torch.from_numpy(b.sqrt_alpha_bar)[t].reshape(-1, 1, 1, 1, 1) * q_ref + \
        torch.from_numpy(b.sqrt_one_minus_alpha_bar)[t].reshape(-1, 1, 1, 1, 1) * nz
    assert torch.allclose(dm.q_sample(lat, t, nz).cpu(), want, atol=1e-6)


def test_attn_cp_decoder_and_quantize(cuda):
    import b200dm
    K, D = 256, 64
    vq = b200dm.VQGAN(num_channels=(32, 64, 128), num_embeddings=K, embedding_dim=D)
    od = OF.AttnCpDecoder(D, 1, (32, 64, 128))
    P = OI.make_params(od.spec(), 5, "stress")
    vq.decoder.set_weights(P)
    cb = OI.codebook(K, D, "KD", seed=3)
    vq.quantizer.set_embeddings(cb)
    z = OI.normal((2, 4, 4, 4, D), 11, 0.05)
    q, idx, perp = vq.quantizer.quantize(z.to(cuda))
    q_ref, idx_ref, perp_ref, _ = OF.quantize(z, cb, "KD")
    assert torch.equal(idx.cpu(), idx_ref) and torch.equal(q.cpu(), q_ref)
    assert abs(perp - perp_ref.item()) <= 1e-3 * perp_ref.item()
    y = vq.decoder(q)
    assert tuple(y.shape) == (2, 16, 16, 16, 1)
    r_e, r_x = rel(y, od.forward(P, q_ref, emu16())), rel(y, od.forward(P, q_ref))
    print(f"attn_cp decoder: rel-L2 vs emu {r_e:.3e}, vs fp32 {r_x:.3e}")
    assert r_e <= tol(8e-3, 1.2e-3) and r_x <= tol(3e-2, 4e-3)


@pytest.mark.parametrize("variant", ["vqgan", "gnorm", "stride"])
@pytest.mark.parametrize("channels", [(32, 64), (16, 32)])
def test_vqgan_family_decoders(cuda, variant, channels):
    """Decoders D2 / D3 / D4 (vqgan.py, vqgan_gnorm.py, vqgan_stride.py; in/out channels 2 as in the main_exp_* scripts) vs
    the oracle: BN folds, GroupNorm + per-voxel PReLU + residual passes, ConvT / conv4+upsample, 2-channel fp32 output with a
    one-group GroupNorm.  (16, 32) exercises the `out < 32` GroupNorm sites.  Same tolerances as the other decoders."""
    import b200dm
    D = 16
    vq = b200dm.VQGAN(in_channels=2, out_channels=2, num_channels=channels, num_res_layers=1, num_res_channels=channels,
                      num_embeddings=64, embedding_dim=D, variant=variant, latent_size=4)
    od = OF.VqganFamilyDecoder(variant, D, 2, channels, 1, channels, 4)
    assert [(n, tuple(s)) for n, s, _ in vq.decoder.spec] == [(n, tuple(s)) for n, s, _ in od.spec()]
    P = OI.make_params(od.spec(), 5, "stress")
    vq.decoder.set_weights(P)
    z = OI.normal((2, 4, 4, 4, D), 11, 0.5)
    y = vq.decoder(z.to(cuda))
    from b200dm import _lib
    assert _lib.debug_flag() == 0
    assert tuple(y.shape) == (2, 16, 16, 16, 2) and y.dtype == torch.float32
    r_e, r_x = rel(y, od.forward(P, z, emu16())), rel(y, od.forward(P, z))
    print(f"{variant} {channels} decoder: rel-L2 vs emu {r_e:.3e}, vs fp32 {r_x:.3e}")
    assert r_e <= tol(1e-2, 1.3e-3) and r_x <= tol(3e-2, 4e-3)


@pytest.mark.parametrize("sampler,cond,S,C_lat,B", [("ddpm", False, 16, 128, 2), ("ddim", False, 16, 128, 2), ("ddpm", True, 32, 256, 2),
                                                     ("ddim", False, 32, 256, 1), ("ddpm", False, 32, 256, 1)])
def test_fused_update_equals_update_kernel(cuda, sampler, cond, S, C_lat, B):
    """The reverse-diffusion update fused into the output conv's epilogue (b200dm_conv_plan_set_fused_update) against the
    stand-alone update kernel on the conv's eps output: same arithmetic, same Philox stream -> bit-identical latents, for the
    DDPM chain down to t = 0 (the noise-free last step) and for a strided DDIM sequence; sharding offset included.  The batch-1
    32^3 x 256 cases are the cfg-4 geometry (one or two tiles per CTA), where unevenly paced epilogue warps exposed a phase slip
    of the fused epilogue's arrive-only barrier; they are repeated to give a rare interleaving a chance."""
    import b200dm
    T = 20
    args = types.SimpleNamespace(timesteps=T, num_gpus=1, kernel_resize=False, bs=B)
    cls = b200dm.ConditionalDiffusionModel if cond else b200dm.DiffusionModel
    dm = cls(S, 256, C_lat, None, args)
    F = 32 if cond else 64
    ou = OUNet(S, C_lat, [64, 128, 256], [False, False, True, True], first_conv_channels=F, conditional=cond)
    P = OI.make_params(ou.spec(), 0, "stress")
    # contraction-scaled output conv: a random-init eps_hat of 10-30x its input would saturate the clip (DDPM) or blow up (DDIM)
    P["out.conv.kernel"] = P["out.conv.kernel"] * 0.05
    dm.network.set_weights(P)
    shape = (B, S, S, S, C_lat)
    x_T = OI.normal(shape, 4321)
    kw = dict(x_T=x_T, seed=99, sample_id0=3, sampler=sampler, last_step=T - 6)
    if sampler == "ddim":
        kw.update(steps=5, last_step=0)
    if cond:
        kw.update(context=torch.arange(B) % 2)
    a = dm.generate(shape, fuse_update=False, **kw)
    assert dm._step["fused"] is False
    from b200dm import _lib
    for _ in range(8 if B == 1 else 1):
        b = dm.generate(shape, fuse_update=True, **kw)
        assert dm._step["fused"] is True, "the output conv of this configuration must take the fused update"
        assert _lib.debug_flag() == 0, "tcgen05 / TMA watchdog"
        assert torch.equal(a, b), (a - b).abs().max().item()
    assert torch.isfinite(a).all() and a.abs().max() > 0.1
    if sampler == "ddpm":   # down to t = 0: the last step adds no noise
        a0 = dm.generate(shape, fuse_update=False, **{**kw, "last_step": 0})
        b0 = dm.generate(shape, **{**kw, "last_step": 0})     # default: fused whenever possible
        assert dm._step["fused"] is True
        assert torch.equal(a0, b0)
        assert not torch.equal(a0, a)
    from b200dm import _lib
    assert _lib.debug_flag() == 0
