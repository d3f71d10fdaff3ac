"""Synthetic datasets of the shapes BASELINE.json names (there is no network for the real
ones): FEMNIST 28x28/62 classes, non-IID CIFAR-10 shards, seq-128 token classification, and
an Occupancy-like 5-feature binary table matching the reference's CSV schema
(python-sdk/data/datatraining.txt: Temperature, Humidity, Light, CO2, HumidityRatio ->
Occupancy; 8143 rows, 21% positive -- SURVEY.md A3).

Every generator is class-conditional (a fixed random prototype per class plus noise) so the
models genuinely learn and committee scores separate honest from Byzantine updates.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch


@dataclass
class Shard:
    x: torch.Tensor          # features (uint8 images / float tables / int64 tokens)
    y: torch.Tensor          # int64 labels
    n_classes: int

    def __len__(self) -> int:
        return int(self.x.shape[0])


def _label_split(n: int, n_classes: int, clients: int, alpha: float, rng: np.random.Generator):
    """Per-client label histograms: alpha == 0 -> IID, else Dirichlet(alpha) skew."""
    if alpha <= 0:
        return [np.full(n_classes, 1.0 / n_classes) for _ in range(clients)]
    return [rng.dirichlet(np.full(n_classes, alpha)) for _ in range(clients)]


def client_sizes(clients: int, mean: int, *, sigma: float, multiple: int = 1, seed: int = 0) -> List[int]:
    """Seeded log-normal shard sizes (unequal clients, as FEMNIST writers are): client i holds a
    multiple of ``multiple`` rows, at least one multiple, and the sizes add up to ``clients`` times
    ``mean`` rounded to a multiple, so a skewed run trains as many samples as an equal one.
    ``sigma = 0`` gives equal sizes."""
    if clients <= 0 or multiple <= 0 or sigma < 0:
        raise ValueError("client_sizes: clients > 0, multiple > 0, sigma >= 0")
    unit = max(int(round(mean / multiple)), 1)                 # per-client mean, in multiples
    total = clients * unit
    z = np.random.default_rng([seed, 7919]).normal(0.0, 1.0, size=clients)
    share = np.exp(sigma * z)
    ideal = share / share.sum() * total
    units = np.maximum(np.floor(ideal), 1).astype(np.int64)
    # largest remainders first up to the total; over it (the one-multiple floor): trim the largest
    frac_order = np.argsort(-(ideal - np.floor(ideal)), kind="stable")
    i = 0
    while units.sum() < total:
        units[frac_order[i % clients]] += 1
        i += 1
    while units.sum() > total and units.max() > 1:
        units[int(np.argmax(units))] -= 1
    return [int(u) * multiple for u in units]


def femnist_like(clients: Optional[int] = None, samples_per_client: Optional[int] = None, *, seed: int = 0,
                 alpha: float = 0.0, n_classes: int = 62, hw: int = 28, noise: float = 48.0,
                 only: Optional[int] = None, sizes: Optional[Sequence[int]] = None) -> List[Shard]:
    """uint8 [n, hw*hw] images: class prototype (0..255) + Gaussian pixel noise.  The class
    prototypes depend only on ``seed``; client ``i``'s samples only on ``(seed, i)``, so a
    rank can generate just its own shard with ``only=i`` (returns a 1-element list).
    ``sizes``: client ``i`` draws ``sizes[i]`` samples instead of ``samples_per_client``
    (``clients`` defaults to ``len(sizes)``); ``alpha > 0`` skews every client's label mix."""
    if sizes is not None:
        sizes = [int(v) for v in sizes]
        if clients is None:
            clients = len(sizes)
        if len(sizes) != clients or any(v <= 0 for v in sizes):
            raise ValueError(f"femnist_like: need {clients} positive sizes, got {sizes}")
    elif clients is None or samples_per_client is None:
        raise ValueError("femnist_like: give clients and samples_per_client, or sizes")
    protos = np.random.default_rng(seed).integers(0, 256, size=(n_classes, hw * hw)).astype(np.float32)
    out = []
    for i in range(clients):
        if only is not None and i != only:
            continue
        n_i = sizes[i] if sizes is not None else samples_per_client
        rng = np.random.default_rng([seed, 1000 + i])
        p = _label_split(n_i, n_classes, 1, alpha, rng)[0]
        y = rng.choice(n_classes, size=n_i, p=p)
        x = protos[y] + rng.normal(0, noise, size=(n_i, hw * hw)).astype(np.float32)
        x = np.clip(x, 0, 255).astype(np.uint8)
        out.append(Shard(torch.from_numpy(x), torch.from_numpy(y.astype(np.int64)), n_classes))
    return out


def cifar_like(clients: int, samples_per_client: int, *, seed: int = 0, alpha: float = 0.5,
               n_classes: int = 10) -> List[Shard]:
    """uint8 [n, 3, 32, 32]; non-IID (Dirichlet) by default, as in config #3/#4."""
    rng = np.random.default_rng(seed)
    protos = rng.integers(0, 256, size=(n_classes, 3, 8, 8)).astype(np.float32)
    protos = np.repeat(np.repeat(protos, 4, axis=2), 4, axis=3)  # blocky 32x32 prototypes
    out = []
    for p in _label_split(samples_per_client, n_classes, clients, alpha, rng):
        y = rng.choice(n_classes, size=samples_per_client, p=p)
        x = protos[y] + rng.normal(0, 40.0, size=(samples_per_client, 3, 32, 32)).astype(np.float32)
        out.append(Shard(torch.from_numpy(np.clip(x, 0, 255).astype(np.uint8)),
                         torch.from_numpy(y.astype(np.int64)), n_classes))
    return out


def tokens_like(clients: int, samples_per_client: int, *, seed: int = 0, seq_len: int = 128,
                vocab: int = 30522, n_classes: int = 2) -> List[Shard]:
    """int64 [n, seq_len] token ids; the label decides which half of the vocabulary the
    sequence is mostly drawn from (sequence classification, BERT config #5)."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(clients):
        y = rng.integers(0, n_classes, size=samples_per_client)
        lo = (y[:, None] * (vocab // n_classes)).astype(np.int64)
        biased = lo + rng.integers(0, vocab // n_classes, size=(samples_per_client, seq_len))
        unif = rng.integers(0, vocab, size=(samples_per_client, seq_len))
        pick = rng.random((samples_per_client, seq_len)) < 0.7
        x = np.where(pick, biased, unif).astype(np.int64)
        out.append(Shard(torch.from_numpy(x), torch.from_numpy(y.astype(np.int64)), n_classes))
    return out


def occupancy_like(n_rows: int = 8143, *, seed: int = 0) -> Tuple[np.ndarray, np.ndarray]:
    """Unnormalised 5-feature table with the reference CSV's ranges (CO2 up to ~2000, Light up
    to ~1500) and ~21% positives; Light and CO2 carry the signal, as in the real data."""
    rng = np.random.default_rng(seed)
    y = (rng.random(n_rows) < 0.2123).astype(np.int64)
    temp = rng.normal(20.6, 1.0, n_rows) + 1.2 * y
    hum = rng.normal(25.7, 5.5, n_rows)
    light = np.where(y == 1, rng.normal(460, 60, n_rows), np.abs(rng.normal(20, 60, n_rows)))
    co2 = np.where(y == 1, rng.normal(1040, 250, n_rows), rng.normal(490, 90, n_rows))
    ratio = rng.normal(0.0039, 0.0008, n_rows)
    x = np.stack([temp, hum, light, co2, ratio], 1).astype(np.float32)
    return x, y
