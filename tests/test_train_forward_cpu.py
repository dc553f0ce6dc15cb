"""CPU checks of the training-mode forward (conditional_dm3d.py:471-499, SURVEY 3.5): the oracle's batch-statistics
BatchNorm against a direct numpy evaluation, the literal loss divisor, and reproducible timestep drawing."""
import types

import numpy as np
import torch

from oracle import init as OI
from oracle import train as OT


def test_batchnorm_train_matches_numpy():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((3, 4, 5, 6, 16)) * rng.uniform(0.1, 5.0, 16) + rng.uniform(-50, 50, 16)
    x[..., 3] = 7.25                              # a constant channel: variance 0, y = beta
    g, b = rng.standard_normal(16), rng.standard_normal(16)
    flat = x.reshape(-1, 16)
    mean = flat.sum(0) / flat.shape[0]
    var = ((flat - mean) ** 2).sum(0) / flat.shape[0]   # biased, as tf.nn.moments
    want = (x - mean) / np.sqrt(var + 1e-3) * g + b
    got = OT.batchnorm_train(torch.from_numpy(x), torch.from_numpy(g), torch.from_numpy(b)).numpy()
    np.testing.assert_allclose(got, want, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(got[..., 3], b[3], atol=1e-9)


def test_training_forward_uses_batch_statistics_not_moving_ones():
    """training=True ignores the moving statistics and couples the samples; training=False is the inference oracle."""
    ou = OT.UNet(8, 8, [64, 128, 256], [False, False, True, True], first_conv_channels=64)
    P = OI.make_params(ou.spec(), 0, "stress")
    x = OI.normal((2, 8, 8, 8, 8), 1)
    t = torch.tensor([3, 30])
    with torch.no_grad():
        y = ou.forward(P, x, t, training=True)
        P2 = {k: (v * 3.0 + 1.0 if k.endswith((".mean", ".var")) else v) for k, v in P.items()}
        assert torch.equal(ou.forward(P2, x, t, training=True), y)
        x2 = x.clone()
        x2[1] = OI.normal((8, 8, 8, 8), 2)
        y2 = ou.forward(P, x2, t, training=True)
        assert (y2[0] - y[0]).norm() > 1e-3 * y[0].norm()
        from oracle.unet import UNet as InferenceUNet
        oi = InferenceUNet(8, 8, [64, 128, 256], [False, False, True, True], first_conv_channels=64)
        assert torch.equal(ou.forward(P, x, t), oi.forward(P, x, t))


def test_literal_loss_divisor():
    """MSE(reduction=SUM)(noise, eps_hat) / (global_bs * lc^4): mean over C, sum over (B, D, H, W), literal divisor."""
    B, S, C, bs = 2, 4, 8, 16
    noise = torch.zeros(B, S, S, S, C, dtype=torch.float64)
    eps = torch.zeros_like(noise)
    eps[..., 0] = 2.0                                  # (n - e)^2 = 4 in one channel of every voxel: mean over C = 4 / C
    assert OT.mse_sum(noise, eps) == B * S ** 3 * 4.0 / C
    assert OT.loss_divisor(bs, C) == bs * C ** 4
    import b200dm
    dm = b200dm.DiffusionModel(S, 256, C, None, types.SimpleNamespace(timesteps=10, num_gpus=1, kernel_resize=False, bs=bs))
    assert dm.loss_divisor() == OT.loss_divisor(bs, C) == 65536.0


def test_timestep_drawing_is_reproducible_from_seed():
    import b200dm
    draw = b200dm.DiffusionModel.draw_timesteps
    a, b = draw(1234, 8, 1000), draw(1234, 8, 1000)
    assert torch.equal(a, b) and a.dtype == torch.int64 and a.shape == (8,)
    assert int(a.min()) >= 0 and int(a.max()) < 1000
    assert not torch.equal(a, draw(1235, 8, 1000))
    big = draw(7, 4096, 10)
    assert set(big.tolist()) == set(range(10))           # U{0..T-1}: every value reachable, none outside
