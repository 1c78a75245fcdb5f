"""DGMR training wrapper with the reference's constructor, hyper-parameters and step semantics
(ref: dgmr/dgmr.py:36-300).  When pytorch_lightning is installed this IS a LightningModule with manual
optimisation, exactly like the reference; without it a minimal stand-in provides the four Lightning
methods the step uses, so the same `training_step` runs under a plain loop (tests / bench).

`training_step` executes the reference's literal schedule (2 discriminator updates + 1 generator update,
whole-generator activation checkpointing, trailing forward).  The leaner, result-equivalent schedule used for
the headline benchmark lives in `skillful_nowcasting_b200.training.gan_step`.
"""
from __future__ import annotations

import torch
from .hub import HubMixin as PyTorchModelHubMixin   # same API; saves compact copies (see hub.py)
from torch.utils.checkpoint import checkpoint

from .common import ContextConditioningStack, LatentConditioningStack
from .discriminators import Discriminator
from .generators import Generator, Sampler
from .losses import GridCellLoss, loss_hinge_disc_both, loss_hinge_gen

try:  # pragma: no cover - not installed in the build image
    import pytorch_lightning as pl

    _Base = pl.LightningModule
    _HAVE_PL = True
except Exception:  # noqa: BLE001
    _HAVE_PL = False

    class _Base(torch.nn.Module):
        """The slice of LightningModule that DGMR.training_step relies on (manual optimisation)."""

        def __init__(self):
            super().__init__()
            self._optimizers = None
            self.logged = {}
            self.hparams = {}

        def save_hyperparameters(self, **kw):
            self.hparams = dict(kw)

        def optimizers(self):
            if self._optimizers is None:
                self._optimizers = self.configure_optimizers()[0]
            return self._optimizers

        def manual_backward(self, loss):
            loss.backward()

        def log_dict(self, d, prog_bar=False):
            self.logged.update({k: v.detach() for k, v in d.items()})


def weight_fn(y, precip_weight_cap=24.0):
    """w(y) = max(y + 1, cap) (ref: dgmr/dgmr.py:20-33).  Kept for API parity; the fused loss kernel applies it."""
    return torch.max(y + 1, torch.tensor(precip_weight_cap, device=y.device))


class DGMR(_Base, PyTorchModelHubMixin, library_name="DGMR",
           tags=["nowcasting", "forecasting", "timeseries", "remote-sensing", "gan"],
           repo_url="https://github.com/openclimatefix/skillful_nowcasting"):
    """Deep Generative Model of Radar (ref: dgmr/dgmr.py:36-130 for the 15 constructor arguments)."""

    def __init__(self, forecast_steps: int = 18, input_channels: int = 1, output_shape: int = 256, gen_lr: float = 5e-5,
                 disc_lr: float = 2e-4, visualize: bool = False, conv_type: str = "standard", num_samples: int = 6,
                 grid_lambda: float = 20.0, beta1: float = 0.0, beta2: float = 0.999, latent_channels: int = 768,
                 context_channels: int = 384, generation_steps: int = 6, precip_weight_cap: float = 24.0):
        super().__init__()
        self.gen_lr, self.disc_lr, self.beta1, self.beta2 = gen_lr, disc_lr, beta1, beta2
        self.grid_regularizer = GridCellLoss(weight_fn=weight_fn, precip_weight_cap=precip_weight_cap)
        self.grid_lambda = grid_lambda
        self.num_samples = num_samples
        self.visualize = visualize
        self.latent_channels, self.context_channels = latent_channels, context_channels
        self.input_channels = input_channels
        self.generation_steps = generation_steps
        self.conditioning_stack = ContextConditioningStack(input_channels=input_channels, conv_type=conv_type,
                                                           output_channels=self.context_channels)
        self.latent_stack = LatentConditioningStack(shape=(8 * self.input_channels, output_shape // 32, output_shape // 32),
                                                    output_channels=self.latent_channels)
        self.sampler = Sampler(forecast_steps=forecast_steps, latent_channels=self.latent_channels,
                               context_channels=self.context_channels)
        self.generator = Generator(self.conditioning_stack, self.latent_stack, self.sampler)
        self.discriminator = Discriminator(input_channels)
        if _HAVE_PL:  # pragma: no cover
            self.save_hyperparameters()
        else:
            self.save_hyperparameters(
                forecast_steps=forecast_steps, input_channels=input_channels, output_shape=output_shape, gen_lr=gen_lr,
                disc_lr=disc_lr, visualize=visualize, conv_type=conv_type, num_samples=num_samples, grid_lambda=grid_lambda,
                beta1=beta1, beta2=beta2, latent_channels=latent_channels, context_channels=context_channels,
                generation_steps=generation_steps, precip_weight_cap=precip_weight_cap)
        self.global_iteration = 0
        self.automatic_optimization = False

    def forward(self, x):
        return self.generator(x)

    def sample(self, x, num_samples=None):
        """Eval-mode ensemble [B,K,T,C,H,W] of K = num_samples (default: the constructor's num_samples) forecasts: Generator.sample."""
        return self.generator.sample(x, self.num_samples if num_samples is None else num_samples)

    # ------------------------------------------------------------------ reference schedule (dgmr/dgmr.py:137-218)
    def _disc_scores(self, images, future_images, predictions):
        generated_sequence = torch.cat([images, predictions], dim=1)
        real_sequence = torch.cat([images, future_images], dim=1)
        return self.discriminator(torch.cat([real_sequence, generated_sequence], dim=0))

    def training_step(self, batch, batch_idx):
        images, future_images = batch
        images, future_images = images.float(), future_images.float()
        self.global_iteration += 1
        g_opt, d_opt = self.optimizers()
        for _ in range(2):  # two discriminator steps per generator step (:148)
            d_opt.zero_grad()
            predictions = checkpoint(self.forward, images, use_reentrant=False)
            discriminator_loss = loss_hinge_disc_both(self._disc_scores(images, future_images, predictions))
            self.manual_backward(discriminator_loss)
            d_opt.step()
        predictions = [checkpoint(self.forward, images, use_reentrant=False) for _ in range(self.generation_steps)]
        from . import ops
        gen_mean = ops.mean_k(predictions)
        grid_cell_reg = self.grid_regularizer(gen_mean, future_images)
        b = images.shape[0]
        generated_scores = [self._disc_scores(images, future_images, p)[b:] for p in predictions]
        generator_disc_loss = loss_hinge_gen(torch.cat(generated_scores, dim=0))
        generator_loss = generator_disc_loss + self.grid_lambda * grid_cell_reg
        g_opt.zero_grad()
        self.manual_backward(generator_loss)
        g_opt.step()
        self.log_dict({"train/d_loss": discriminator_loss, "train/g_loss": generator_loss, "train/grid_loss": grid_cell_reg},
                      prog_bar=True)
        generated_images = self(images)  # the reference always runs this trailing forward (:213)
        return generated_images

    def validation_step(self, batch, batch_idx):
        images, future_images = batch
        images, future_images = images.float(), future_images.float()
        from . import ops
        for _ in range(2):
            discriminator_loss = loss_hinge_disc_both(self._disc_scores(images, future_images, self(images)))
        predictions = [self(images) for _ in range(self.generation_steps)]
        grid_cell_reg = self.grid_regularizer(ops.mean_k(predictions), future_images)
        b = images.shape[0]
        generated_scores = [self._disc_scores(images, future_images, p)[b:] for p in predictions]
        generator_loss = loss_hinge_gen(torch.cat(generated_scores, dim=0)) + self.grid_lambda * grid_cell_reg
        self.log_dict({"val/d_loss": discriminator_loss, "val/g_loss": generator_loss, "val/grid_loss": grid_cell_reg},
                      prog_bar=True)

    def configure_optimizers(self):
        """Adam(lr, betas=(beta1, beta2)) for G and D (ref: dgmr/dgmr.py:292-300), stepping through the fused
        Adam kernel of the C ABI."""
        from .training import Adam

        opt_g = Adam(self.generator.parameters(), lr=self.gen_lr, betas=(self.beta1, self.beta2))
        opt_d = Adam(self.discriminator.parameters(), lr=self.disc_lr, betas=(self.beta1, self.beta2))
        return [opt_g, opt_d], []
