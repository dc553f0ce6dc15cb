"""Training-mode forward of the 3D latent U-Net and train_step's loss (oracle; test infrastructure only).

  network([x_t, t, ctx], training=True)                 conditional_dm3d.py:493 (SURVEY 3.5)
  loss = MSE(reduction=SUM)(noise, eps_hat) / (global_bs * lc^4)   conditional_dm3d.py:496-499

With ``training=True`` every keras BatchNormalization normalises with the mean and biased variance of the current batch
over every axis but the channels (tf.nn.moments); the moving statistics are neither used nor updated here.  The
inference-mode oracle (``oracle.unet.UNet``) is unchanged: this module subclasses it.
"""
from __future__ import annotations

import torch

from . import ops
from .ops import Emu, EXACT
from .unet import UNet as _UNet


def batchnorm_train(x, gamma, beta, eps: float = 1e-3):
    """keras BatchNormalization, training=True: per-channel mean / biased variance of this batch, then the inference
    formula (ops.batchnorm_infer) with those statistics."""
    dims = tuple(range(x.dim() - 1))
    mean = x.mean(dim=dims)
    var = x.var(dim=dims, unbiased=False)
    return ops.batchnorm_infer(x, gamma, beta, mean, var, eps)


class UNet(_UNet):
    """oracle.unet.UNet with ``forward(..., training=True)``.  A concat [x | skip] is normalised per channel, so its
    statistics are those of each half's own tensor."""

    training = False

    def _bn_apply(self, P, name, x):
        if self.training:
            return batchnorm_train(x, P[f"{name}.gamma"], P[f"{name}.beta"])
        return super()._bn_apply(P, name, x)

    def forward(self, P, x, t, ctx=None, emu: Emu = EXACT, training=False):
        self.training = bool(training)
        try:
            return super().forward(P, x, t, ctx=ctx, emu=emu)
        finally:
            self.training = False


def loss_divisor(global_bs, lc):
    """conditional_dm3d.py:496-499 divides by global_bs * lc^4 (lc = latent channels): not the element count."""
    return global_bs * lc ** 4


def mse_sum(noise, eps_hat):
    """keras MeanSquaredError(reduction=SUM): mean over the last axis, summed over every other position (fp64)."""
    return ((noise.double() - eps_hat.double()) ** 2).mean(dim=-1).sum().item()


def q_sample(betas, latents, t, noise):
    """x_t = sqrt(abar_t) z + sqrt(1 - abar_t) noise (conditional_dm3d.py:484-490), fp32 tables, fp32 op order."""
    idx = torch.as_tensor(t).long()
    sqb = torch.from_numpy(betas.sqrt_alpha_bar)[idx].reshape(-1, 1, 1, 1, 1)
    osqb = torch.from_numpy(betas.sqrt_one_minus_alpha_bar)[idx].reshape(-1, 1, 1, 1, 1)
    return sqb * latents.float() + osqb * noise.float()


def train_loss(unet: UNet, P, betas, latents, t, noise, global_bs, ctx=None, emu: Emu = EXACT):
    """train_step's loss without the gradient step (conditional_dm3d.py:471-499): q-sample, training-mode eps_hat, loss."""
    eps = unet.forward(P, q_sample(betas, latents, t, noise), torch.as_tensor(t).long(), ctx=ctx, emu=emu, training=True)
    return mse_sum(noise, eps) / loss_divisor(global_bs, latents.shape[-1])
