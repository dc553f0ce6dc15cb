"""GPU checks of the training-mode forward: batch-statistics BatchNorm kernel, network(..., training=True) against the
oracle's training mode, the q-sample and loss kernels and DiffusionModel.train_loss (conditional_dm3d.py:471-499).

Tolerances: the statistics kernel reduces in fp32 partials / fp64 combine on the same 16-bit input as the fp64 reference, so
scale and shift agree to ~1e-6 relative.  Training-mode eps_hat goes through the same ~100 16-bit storage points as the
inference forward and is held to the same storage-floor bounds (tests/test_model_gpu.py, DESIGN.md section 2).
"""
import os
import types

import numpy as np
import pytest
import torch

from oracle import init as OI, philox
from oracle import train as OT
from oracle.ops import Emu
from oracle.schedule import Betas as OBetas

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-20)).item()


def tol(bf16, fp16):
    from b200dm import _lib
    return bf16 if _lib.precision() == "bf16" else fp16


def emu16():
    from b200dm import _lib
    return Emu(True, dtype=_lib.ACT_DTYPE)


def flag_ok():
    from b200dm import _lib
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0


@pytest.mark.parametrize("C,rows", [(8, 1000), (16, 4096), (32, 8 * 32 ** 3), (64, 8 * 32 ** 3), (128, 8 * 16 ** 3),
                                    (256, 8 * 8 ** 3), (512, 8 * 8 ** 3), (96, 5000)])
def test_bn_stats_against_fp64(cuda, C, rows):
    from b200dm import _lib, ops
    if 256 % (C // 8):
        with pytest.raises(_lib.B200dmError):
            ops.bn_stats(torch.zeros(rows, C, dtype=_lib.ACT_DTYPE, device=cuda), torch.ones(C, device=cuda), torch.zeros(C, device=cuda))
        return
    g = torch.Generator(device="cpu").manual_seed(C)
    x = torch.randn(rows, C, generator=g) * torch.rand(C, generator=g) * 3 + torch.randn(C, generator=g)
    x[:, 0] = 0.3                                        # constant channel: var = 0
    x[:, 1] = 300.0 + 2.0 * torch.randn(rows, generator=g)   # |mean| >> std: Sigma x^2 - (Sigma x)^2 would cancel
    x16 = x.to(_lib.ACT_DTYPE).to(cuda)
    gam, bet = torch.randn(C, generator=g).to(cuda), torch.randn(C, generator=g).to(cuda)
    sc, sh = ops.bn_stats(x16, gam, bet)
    sc2, sh2 = ops.bn_stats(x16, gam, bet)
    assert torch.equal(sc, sc2) and torch.equal(sh, sh2), "not bit-reproducible"
    xd = x16.double().cpu()
    m, v = xd.mean(0), xd.var(0, unbiased=False)
    s_ref = gam.double().cpu() / torch.sqrt(v + 1e-3)
    h_ref = bet.double().cpu() - m * s_ref
    es = ((sc.double().cpu() - s_ref).abs() / s_ref.abs()).max().item()
    eh = ((sh.double().cpu() - h_ref).abs() / (bet.double().cpu().abs() + (m * s_ref).abs())).max().item()
    print(f"bn_stats C={C} rows={rows}: max rel err scale {es:.2e} shift {eh:.2e}")
    assert es <= 5e-6 and eh <= 5e-6, (es, eh)


def _unet_pair(S, C_lat, cond, seed=0):
    import b200dm
    F = 32 if cond else 64
    net = b200dm.build_model(S, C_lat, [64, 128, 256], [False, False, True, True], context_dim=1 if cond else None)
    ou = OT.UNet(S, C_lat, [64, 128, 256], [False, False, True, True], first_conv_channels=F, conditional=cond)
    P = OI.make_params(ou.spec(), seed, "stress")
    # moving statistics far from the batch's: a training forward that read them would miss the oracle by O(1)
    for k in P:
        if k.endswith(".mean"):
            P[k] = P[k] + 0.5
        elif k.endswith(".var"):
            P[k] = P[k] * 2.0 + 0.5
    net.set_weights(P)
    return net, ou, P


@pytest.mark.parametrize("cond", [False, True])
def test_training_forward_8cubed(cuda, cond):
    S, C_lat, B = 8, 16 if cond else 8, 2
    net, ou, P = _unet_pair(S, C_lat, cond)
    net.compile(B, 50)
    x = OI.normal((B, S, S, S, C_lat), 1)
    tt = torch.tensor([37, 5])
    ctx = torch.tensor([0, 1]) if cond else None
    inp = [x.to(cuda), tt] + ([ctx] if cond else [])
    y_inf = net(inp)
    y = net(inp, training=True)
    flag_ok()
    with torch.no_grad():
        ref_e = ou.forward(P, x, tt, ctx=ctx, emu=emu16(), training=True)
        ref_x = ou.forward(P, x, tt, ctx=ctx, training=True)
    r_e, r_x = rel(y, ref_e), rel(y, ref_x)
    print(f"training eps_hat 8^3 cond={cond}: rel-L2 vs emulating oracle {r_e:.3e}, vs fp32 oracle {r_x:.3e}")
    assert r_e <= 2.5e-2 and r_x <= 2.5e-2, (r_e, r_x)
    assert rel(y, y_inf) > 0.1, "training mode must not use the moving statistics"
    # inference eps_hat is bit-identical before and after a training-mode call
    assert torch.equal(net(inp), y_inf)
    # coupling: in training mode sample 1 changes sample 0's eps_hat; in inference mode it does not
    x2 = x.clone()
    x2[1] = OI.normal((S, S, S, C_lat), 2)
    inp2 = [x2.to(cuda), tt] + ([ctx] if cond else [])
    assert rel(net(inp2, training=True)[0], y[0]) > 1e-3
    assert torch.equal(net(inp2)[0], y_inf[0])
    assert torch.equal(net(inp, training=True), y), "training forward not bit-reproducible"


def test_training_forward_cfg2(cuda):
    """cfg-2: conditional U-Net, B=8, 32^3 x 256, per-sample t and class ids, training=True vs the fp32 oracle."""
    import b200dm
    torch.set_num_threads(os.cpu_count() or 1)
    net = b200dm.build_model(32, 256, [64, 128, 256], [False, False, True, True], context_dim=1)
    ou = OT.UNet(32, 256, [64, 128, 256], [False, False, True, True], first_conv_channels=32, conditional=True)
    P = OI.make_params(ou.spec(), 0, "stress")
    net.set_weights(P)
    B = 8
    net.compile(B, 1000)
    x = OI.normal((B, 32, 32, 32, 256), 1)
    ctx = torch.arange(B) % 2
    tt = torch.tensor([999, 500, 3, 250, 750, 0, 100, 900])
    y = net([x.to(cuda), tt, ctx], training=True).cpu()
    flag_ok()
    with torch.no_grad():
        ref = ou.forward(P, x, tt, ctx=ctx, training=True)
    r = rel(y, ref)
    print(f"training eps_hat cfg-2 B=8: rel-L2 vs fp32 oracle {r:.3e}, max-abs {(y - ref).abs().max().item():.3e}")
    assert r <= tol(2.5e-2, 4e-3), r


def test_q_sample_kernel(cuda):
    import b200dm
    from b200dm import _lib
    B, S, C, T = 3, 4, 8, 50
    dm = b200dm.DiffusionModel(S, 64, C, None, types.SimpleNamespace(timesteps=T, num_gpus=1, kernel_resize=False, bs=B))
    z, nz = OI.normal((B, S, S, S, C), 13), OI.normal((B, S, S, S, C), 14)
    t = torch.tensor([0, 17, 49])
    ob = OBetas(T)
    sqb = torch.from_numpy(ob.sqrt_alpha_bar)[t].reshape(-1, 1, 1, 1, 1)
    osqb = torch.from_numpy(ob.sqrt_one_minus_alpha_bar)[t].reshape(-1, 1, 1, 1, 1)
    host = sqb * z + osqb * nz                        # the former host helper's formula
    assert torch.equal(dm.q_sample(z.to(cuda), t, nz).cpu(), host)
    # Philox stream 2 (the sampler's streams are 0 and 1), keyed by (seed, global sample index, element)
    dm.b.to(cuda)
    t_dev = t.to(torch.int32).to(cuda)
    x16, x32 = b200dm.ops.q_sample(dm.b, z.to(cuda), t_dev, seed=99, sample_id0=5, want_f32=True)
    n = torch.from_numpy(philox.normal(99, 0, np.arange(5, 5 + B), S ** 3 * C, stream=2)).reshape(z.shape)
    assert (x32.cpu() - (sqb * z + osqb * n)).abs().max().item() <= 1e-5
    assert torch.equal(x16, x32.to(_lib.ACT_DTYPE))
    x32b = b200dm.ops.q_sample(dm.b, z[1:].contiguous().to(cuda), t_dev[1:], seed=99, sample_id0=6, want_f32=True)[1]
    assert torch.equal(x32b, x32[1:]), "noise must depend on the global sample index only"


def test_noise_loss_kernel(cuda):
    from b200dm import ops
    B, S, C = 2, 8, 16
    eps, nz = OI.normal((B, S, S, S, C), 3), OI.normal((B, S, S, S, C), 4)
    got = ops.noise_loss(eps.to(cuda), 7.0, noise=nz.to(cuda)).item()
    want = OT.mse_sum(nz, eps) / 7.0
    assert abs(got - want) <= 1e-6 * want
    n = torch.from_numpy(philox.normal(5, 0, np.arange(B), S ** 3 * C, stream=2)).reshape(eps.shape)
    got = ops.noise_loss(eps.to(cuda), 7.0, seed=5).item()
    assert abs(got - OT.mse_sum(n, eps) / 7.0) <= 1e-5 * got
    assert ops.noise_loss(eps.to(cuda), 7.0, seed=5).item() == got


@pytest.mark.parametrize("cond", [False, True])
def test_train_loss(cuda, cond):
    import b200dm
    S, C, B, T = 8, 8, 2, 50
    cls = b200dm.ConditionalDiffusionModel if cond else b200dm.DiffusionModel
    dm = cls(S, 64, C, None, types.SimpleNamespace(timesteps=T, num_gpus=1, kernel_resize=False, bs=4))
    ou = OT.UNet(S, C, [64, 128, 256], [False, False, True, True], first_conv_channels=cls.first_conv_channels, conditional=cond)
    P = OI.make_params(ou.spec(), 0, "stress")
    P["out.conv.kernel"] = P["out.conv.kernel"] * 0.05   # eps_hat of the size of the noise: the loss is not dominated by eps_hat alone
    dm.network.set_weights(P)
    z = OI.normal((B, S, S, S, C), 21, 0.5)
    nz = OI.normal((B, S, S, S, C), 22)
    t = torch.tensor([7, 42])
    ctx = torch.tensor([1, 0]) if cond else None
    got = dm.train_loss(latents=z.to(cuda), t=t, noise=nz, context=ctx).item()
    flag_ok()
    with torch.no_grad():
        want = OT.train_loss(ou, P, OBetas(T), z, t, nz, 4, ctx=ctx, emu=emu16())
    print(f"train_loss cond={cond}: {got:.6e} vs oracle {want:.6e} (rel {abs(got - want) / want:.2e})")
    assert abs(got - want) <= 1e-3 * want, (got, want)
    assert torch.equal(dm.last_t, t)
    # without injection: t from the seeded host generator, noise from Philox stream 2 -> bit-reproducible from seed
    a = dm.train_loss(latents=z.to(cuda), seed=11, context=ctx)
    assert torch.equal(dm.last_t, b200dm.DiffusionModel.draw_timesteps(11, B, T)) and dm.last_seed == 11
    b = dm.train_loss(latents=z.to(cuda), seed=11, context=ctx)
    c = dm.train_loss(latents=z.to(cuda), seed=12, context=ctx)
    assert a.dtype == torch.float32 and a.dim() == 0
    assert torch.equal(a, b) and not torch.equal(a, c)
    n = torch.from_numpy(philox.normal(11, 0, np.arange(B), S ** 3 * C, stream=2)).reshape(z.shape)
    want11 = OT.train_loss(ou, P, OBetas(T), z, b200dm.DiffusionModel.draw_timesteps(11, B, T), n, 4, ctx=ctx, emu=emu16())
    assert abs(a.item() - want11) <= 1e-3 * want11, (a.item(), want11)
