"""Measurement simulation ``y = A x + white noise`` (reference src/physics/simulation.py:12-74) and low-dose
Poisson data with its statistical weights (:func:`simulate_poisson`)."""
from typing import Any, Iterator, Optional, Tuple

import numpy as np
import torch
from torch import Tensor


def simulate(x: Tensor, ray_trafo, white_noise_rel_stddev: float, rng=None,
             return_noise_level: bool = False):
    """Noise level = ``rel_stddev * mean|A x|``; the noise comes from a numpy generator (pass a
    seeded one for reproducibility), as in the reference (:12-23).

    The reference reads the noise level back to the host (``.item()``) before it draws
    ``rng.normal(scale=noise_level)``.  numpy forms that draw as ``scale * standard_normal`` in
    float64, so here the standard-normal field is drawn first and scaled on the device by the
    float64 noise level: same random stream, same values, and no host synchronisation between the
    projection and the noise (the level is only read back when ``return_noise_level`` asks for it)."""
    observation = ray_trafo(x)
    if rng is None:
        rng = np.random.default_rng()
    noise_level = white_noise_rel_stddev * torch.mean(torch.abs(observation)).to(torch.float64)
    z = torch.from_numpy(rng.standard_normal(size=tuple(observation.shape)))
    noise = (z.to(observation.device) * noise_level).to(dtype=observation.dtype)
    noisy_observation = observation + noise
    return (noisy_observation, noise_level.item()) if return_noise_level else noisy_observation


def simulate_poisson(x: Tensor, ray_trafo, photons: float, mu: float, rng: np.random.Generator,
                     min_count: float = 0.1):
    """Low-dose transmission data: photon counts ``N ~ Poisson(photons * exp(-mu * A x))`` per detector bin, the
    log-transformed line integrals ``y = -log(max(N, min_count) / photons) / mu`` and their statistical weights.

    ``mu`` scales the image to attenuation per unit length of the geometry; ``min_count`` replaces empty bins before
    the log (a bin that saw no photon has no finite line integral).  After the log the variance of a bin is about
    ``1 / (mu^2 N)``, so the penalised weighted least-squares weights are ``W = max(N, min_count)``, returned
    normalised to mean 1 per sample so that ``gamma`` keeps its meaning.  The counts are drawn on the host from the
    numpy generator ``rng`` (pass a seeded one for reproducible data): one read-back of ``A x``, outside any sampling
    loop.  Returns ``(y, W)``, float32 of ``A x``'s shape on ``x``'s device; pass ``W`` as ``weights=`` to the
    data-consistency calls (:class:`~.b200_ray_trafo.MeasurementWeights`)."""
    if not (photons > 0 and mu > 0 and min_count > 0):
        raise ValueError('simulate_poisson: photons, mu and min_count must be > 0')
    ax = ray_trafo(x)
    lam = float(photons) * np.exp(-float(mu) * ax.detach().to(torch.float64).cpu().numpy())
    counts = np.maximum(rng.poisson(lam), float(min_count))
    y = -np.log(counts / float(photons)) / float(mu)
    per_sample = counts.reshape(counts.shape[0], -1).mean(axis=1).reshape(-1, *([1] * (counts.ndim - 1)))
    w = counts / per_sample
    dev = ax.device
    return (torch.from_numpy(y).to(device=dev, dtype=torch.float32),
            torch.from_numpy(w).to(device=dev, dtype=torch.float32))


class SimulatedDataset(torch.utils.data.Dataset):
    """Lazily simulated measurements of an image dataset: item ``k`` is the triple
    ``(y_k, x_k, fbp(y_k))`` with ``y_k = simulate(x_k)`` (contract of the reference class,
    src/physics/simulation.py:25-74, which the drivers iterate and index).

    Noise is reproducible per item: unless a generator is shared across items (``rng``), item ``k`` draws from
    ``numpy.random.default_rng(use_fixed_seeds_starting_from + k)`` (``None`` = fresh entropy); passing both a
    generator and a seed base is refused like in the reference."""

    def __init__(self, image_dataset, ray_trafo, white_noise_rel_stddev: float,
                 use_fixed_seeds_starting_from: Optional[int] = 1,
                 rng: Optional[np.random.Generator] = None, device: Optional[Any] = None):
        super().__init__()
        assert rng is None or use_fixed_seeds_starting_from is None, \
            'must not use fixed seeds when passing a custom rng'
        self.image_dataset, self.ray_trafo, self.device = image_dataset, ray_trafo, device
        self.white_noise_rel_stddev = white_noise_rel_stddev
        self.use_fixed_seeds_starting_from, self.rng = use_fixed_seeds_starting_from, rng

    def _rng_for(self, k: int) -> np.random.Generator:
        if self.rng is not None:
            return self.rng
        base = self.use_fixed_seeds_starting_from
        return np.random.default_rng(base + k if base is not None else None)

    def _triple(self, k: int, image: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        image = image.to(device=self.device)
        y = simulate(image.unsqueeze(0), self.ray_trafo, self.white_noise_rel_stddev, rng=self._rng_for(k))
        y = y.to(device=self.device)
        return y[0], image, self.ray_trafo.fbp(y)[0].to(device=self.device)

    def __len__(self):
        return len(self.image_dataset)

    def __getitem__(self, k: int) -> Tuple[Tensor, Tensor, Tensor]:
        return self._triple(k, self.image_dataset[k])

    def __iter__(self) -> Iterator[Tuple[Tensor, Tensor, Tensor]]:
        return (self._triple(k, image) for k, image in enumerate(self.image_dataset))
