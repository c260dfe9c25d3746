"""Shared plumbing of the VAE / GMVAE model classes: lazy engine construction and the run_model
call (the reference builds its TF graph at this point; we bind device buffers instead)."""
from __future__ import annotations

from typing import Optional

import torch

from .engine import Engine


class _EngineBacked:
    _model_kind = "gmvae"

    def _engine_kwargs(self) -> dict:
        raise NotImplementedError

    def _init_backing(self, precision: str = "bf16", objective: str = "reference", learning_rate: float = 1e-3,
                      max_batch: Optional[int] = None, device: Optional[int] = None, deterministic: bool = False):
        self._precision, self._objective = precision, objective
        self._deterministic = deterministic
        self._learning_rate, self._max_batch, self._device = learning_rate, max_batch, device
        self._engine: Optional[Engine] = None

    def configure(self, precision: Optional[str] = None, objective: Optional[str] = None,
                  learning_rate: Optional[float] = None, max_batch: Optional[int] = None, device: Optional[int] = None,
                  deterministic: Optional[bool] = None):
        """Additive knobs with no reference counterpart (precision / objective / optimiser lr / bitwise-reproducible steps)."""
        if self._engine is not None:
            raise RuntimeError("configure() must be called before the first run_model()")
        if precision is not None: self._precision = precision
        if objective is not None: self._objective = objective
        if learning_rate is not None: self._learning_rate = learning_rate
        if max_batch is not None: self._max_batch = max_batch
        if device is not None: self._device = device
        if deterministic is not None: self._deterministic = bool(deterministic)
        return self

    def engine(self, batch: Optional[int] = None) -> Engine:
        if self._engine is None:
            mb = self._max_batch or batch
            if mb is None:
                raise RuntimeError("engine not built yet: call run_model() or configure(max_batch=...)")
            kw = self._engine_kwargs()
            self._engine = Engine(precision=self._precision, objective=self._objective, max_batch=int(mb),
                                  learning_rate=self._learning_rate, device=self._device,
                                  seed=self.random_seed, deterministic=self._deterministic, **kw)
        return self._engine

    def _run(self, images, targets, eps, gumbel_u) -> torch.Tensor:
        if targets is not images:
            if tuple(targets.shape) != tuple(images.shape) or not bool((torch.as_tensor(targets) == torch.as_tensor(images)).all()):
                raise NotImplementedError("targets must equal images (the reference always passes the same tensor, runners.py:130-134)")
        B = images.shape[0]
        eng = self.engine(B)
        loss = eng.forward_backward(images, eps=eps, gumbel_u=gumbel_u)
        return loss[0]

    # ---- inference helpers shared by VAE and GMVAE -----------------------------------------------
    def _noise_gen(self):
        g = getattr(self, "_gen", None)
        if g is None:
            g = torch.Generator(device="cpu")
            g.manual_seed(self.random_seed if self.random_seed is not None else torch.seed() % (2 ** 31))
            self._gen = g
        return g

    def _randn(self, *shape):
        return torch.randn(*shape, generator=self._noise_gen())

    def reconstruct_images(self, images):
        """Bernoulli means of p(x|z) with z ~ q(z|x[,y]) (gmvae.py:109-121, vae.py:80-88)."""
        eng = self.engine(images.shape[0])
        _, _, z = eng.encode(images)
        return eng.decode(z)

    def generate_sample_images(self, z=None, num_samples=1, name="sample_images"):
        """Bernoulli means for given latent points, or for prior samples (gmvae.py:124-137, vae.py:91-102)."""
        if z is None:
            z = self.generate_samples(num_samples)
        return self.engine().decode(z)

    # scalar summaries of the reference (`nll_scalar`, `kl_div_z`, `nent`, `elbo`)
    def summaries(self) -> dict:
        t = self.engine().loss_buf.detach().cpu()
        out = {"nll_scalar": float(t[1]), "kl_div_z": float(t[2]), "elbo": -float(t[0])}
        if self._model_kind == "gmvae":
            out["nent"] = float(t[3])
        return out
