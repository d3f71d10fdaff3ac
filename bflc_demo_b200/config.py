"""One runtime configuration object shared by Python and the C++ ledger.

The reference hard-codes its protocol constants twice and keeps them in sync by hand:
C++ ``#define``s (CommitteePrecompiled.h:4-19) and Python module globals
(python-sdk/main.py:52,62,65,68-69,87-88) -- changing the committee size means recompiling
the blockchain node (SURVEY.md 5.6).  Here there is exactly one validated dataclass; the
C++ side receives it through ``to_ledger_config``.
"""
from __future__ import annotations

import dataclasses
import json
import math
import os
from dataclasses import dataclass, field
from typing import List, Optional

SERVER_OPTIMIZERS = ("none", "momentum", "adam", "yogi")


@dataclass
class FLConfig:
    # ---- protocol (reference names in comments) ----
    clients: int = 20                 # CLIENT_NUM            H:17 / M:52
    committee_size: int = 4           # COMM_COUNT            H:11
    aggregate_count: int = 6          # AGGREGATE_COUNT       H:13
    needed_updates: int = 10          # NEEDED_UPDATE_COUNT   H:15
    learning_rate: float = 0.001      # learning_rate         H:19 / M:88
    max_epoch: int = 1000             # MAX_EPOCH             M:65
    weight_by_score: bool = False     # False = reference (scores filter, n_samples weight)
    solo: bool = False                # every client trains and scores (single-GPU runs)
    seed: int = 0
    # ---- model / data ----
    model: str = "mlp"                # softmax | mlp | lenet5 | resnet18 | bert
    dataset: str = "femnist"          # occupancy | femnist | cifar10 | tokens
    hidden: int = 256                 # MLP hidden width
    batch_size: int = 100             # M:87
    local_epochs: int = 1             # one pass per round (M:141-148)
    samples_per_client: int = 300     # ~ 6107 / 20 in the reference split (A3)
    val_samples: int = 0              # 0 = validate on the whole shard (M:191)
    optimizer: str = "sgd"            # sgd (M:127) | adam (commented alternative, M:126)
    dtype: str = "bf16"               # fp32 | bf16 | fp8
    non_iid_alpha: float = 0.0        # 0 = IID contiguous split (M:43-48); >0 Dirichlet skew
    # ---- drift under skewed data (MultiClientEngine only; the other engines refuse them) ----
    prox_mu: float = 0.0              # FedProx: local loss + mu/2 ||w - w_global||^2
    server_optimizer: str = "none"    # none (FedAvg) | momentum (FedAvgM) | adam (FedAdam) | yogi (FedYogi)
    server_lr: float = 1.0            # server step on the pseudo-gradient (average - global)
    server_beta1: float = 0.9
    server_beta2: float = 0.99
    server_tau: float = 1e-3          # adaptivity; the second moment starts at tau^2
    # ---- faults (SURVEY.md 5.3) ----
    byzantine_ranks: List[int] = field(default_factory=list)
    byzantine_scale: float = 5.0
    straggler_ranks: List[int] = field(default_factory=list)   # these clients publish late ...
    straggler_delay_us: int = 0                                # ... by this much (first-K-wins test)
    # ---- engine ----
    backend: str = "auto"             # auto | fused (P2P kernels) | nccl (baseline) | gloo
    two_shot: Optional[bool] = None   # None = by model size
    use_multicast: bool = True
    stage_candidates: bool = True     # committee pulls each candidate's weights once (P2P) vs
                                      # the validation GEMMs TMA-loading peers' HBM directly
    cuda_graph: bool = True
    fused_step: bool = True           # MLP: all local steps of a round in one persistent kernel
    ring_slots: int = 256

    def validate(self) -> "FLConfig":
        c = self
        if c.clients < 1:
            raise ValueError("clients must be >= 1")
        if c.committee_size < 1:
            raise ValueError("committee_size must be >= 1")
        if c.aggregate_count < 1 or c.aggregate_count > c.needed_updates:
            raise ValueError("need 1 <= aggregate_count <= needed_updates")
        if c.solo:
            if c.committee_size > c.clients or c.needed_updates > c.clients:
                raise ValueError("solo: committee_size and needed_updates must be <= clients")
        else:
            # implied (never checked) by the reference: NEEDED <= CLIENT - COMM.  The reference also
            # has COMM <= NEEDED (H:11-15); a committee larger than the trainer set (BASELINE.json
            # config #4: committee 5 of 8) is allowed here: re-election takes every scored
            # trainer and refills from the outgoing committee (consensus_math.hpp step 5).
            if c.needed_updates > c.clients - c.committee_size:
                raise ValueError("needed_updates > clients - committee_size: not enough trainers")
        if not (c.learning_rate > 0):
            raise ValueError("learning_rate must be > 0")
        if c.optimizer not in ("sgd", "adam"):
            raise ValueError("optimizer must be sgd or adam")
        if c.dtype not in ("fp32", "bf16", "fp8"):
            raise ValueError("dtype must be fp32, bf16 or fp8")
        for r in c.byzantine_ranks:
            if not (0 <= r < c.clients):
                raise ValueError(f"byzantine rank {r} out of range")
        if not (math.isfinite(c.prox_mu) and c.prox_mu >= 0):
            raise ValueError("prox_mu must be finite and >= 0")
        if c.server_optimizer not in SERVER_OPTIMIZERS:
            raise ValueError("server_optimizer must be one of " + ", ".join(SERVER_OPTIMIZERS))
        if not (c.server_lr > 0 and math.isfinite(c.server_lr)):
            raise ValueError("server_lr must be > 0")
        for name in ("server_beta1", "server_beta2"):
            if not (0 <= getattr(c, name) < 1):
                raise ValueError(f"{name} must be in [0, 1)")
        if not (c.server_tau > 0 and math.isfinite(c.server_tau)):
            raise ValueError("server_tau must be > 0")
        return self

    @property
    def plain_fedavg(self) -> bool:
        """No proximal term and no server optimizer: the update rule of every engine."""
        return self.prox_mu == 0 and self.server_optimizer == "none"

    def require_plain_fedavg(self, engine: str) -> None:
        """FedProx and the server optimizers exist in MultiClientEngine only; the other engines
        refuse them rather than train something else than what was asked for."""
        if not self.plain_fedavg:
            raise ValueError(f"{engine} supports neither prox_mu > 0 nor a server optimizer "
                             f"(prox_mu={self.prox_mu}, server_optimizer={self.server_optimizer!r}); "
                             "use MultiClientEngine (run.py --clients N)")

    @property
    def n_trainers(self) -> int:
        return self.clients if self.solo else self.clients - self.committee_size

    def to_ledger_config(self, model_size: int):
        from ._native import ledger

        L = ledger()
        lc = L.LedgerConfig()
        lc.client_num = self.clients
        lc.comm_count = self.committee_size
        lc.aggregate_count = self.aggregate_count
        lc.needed_update_count = self.needed_updates
        lc.learning_rate = self.learning_rate
        lc.model_size = int(model_size)
        lc.weight_by_score = 1 if self.weight_by_score else 0
        lc.solo = 1 if self.solo else 0
        lc.seed = self.seed
        err = lc.validate()
        if err:
            raise ValueError(err)
        return lc

    # ---- construction helpers -------------------------------------------------
    @classmethod
    def reference_default(cls) -> "FLConfig":
        """The reference's own constants: 20 clients, 4 committee, top-6 of 10, lr 1e-3,
        softmax regression 5->2 on UCI Occupancy (H:7-19, M:52-69)."""
        return cls(model="softmax", dataset="occupancy").validate()

    @classmethod
    def reference_scaled(cls, clients: int, **kw) -> "FLConfig":
        """The reference's 20/4/10/6 proportions scaled to another client count."""
        if clients == 20:
            base = dict()
        else:
            comm = max(1, clients // 5)
            trainers = clients - comm
            needed = max(comm, (trainers * 10 + 15) // 16)
            agg = max(1, min(needed, max(comm, (needed * 6 + 9) // 10)))
            base = dict(clients=clients, committee_size=comm, needed_updates=needed,
                        aggregate_count=agg)
        base.update(dict(model="softmax", dataset="occupancy"))
        base.update(kw)
        return cls(**base).validate()

    @classmethod
    def for_world(cls, n: int, committee_size: Optional[int] = None,
                  needed_updates: Optional[int] = None, **kw) -> "FLConfig":
        """The benchmark family of BASELINE.json: n clients, committee 3 at n=8, 2 at n=4,
        1 at n=2, solo at n=1 (``committee_size=5`` gives config #4); by default every trainer's
        update is needed (``needed_updates=k`` < trainers enables first-k-wins admission);
        top-(needed-1) aggregated (at least the committee size when that many are admitted)."""
        if n == 1:
            base = dict(clients=1, committee_size=1, needed_updates=1, aggregate_count=1, solo=True)
        else:
            comm = committee_size or {2: 1, 4: 2, 8: 3}.get(n, max(1, n // 3))
            if not (1 <= comm < n):
                raise ValueError(f"committee_size must be in [1, {n - 1}] for {n} clients")
            trainers = n - comm
            needed = min(needed_updates or trainers, trainers)
            base = dict(clients=n, committee_size=comm, needed_updates=needed,
                        aggregate_count=min(max(comm if comm <= needed else 1, needed - 1, 1), needed))
        base.update(kw)
        return cls(**base).validate()

    @classmethod
    def from_json(cls, text: str) -> "FLConfig":
        return cls(**json.loads(text)).validate()

    @classmethod
    def from_env(cls, prefix: str = "BFLC_", **defaults) -> "FLConfig":
        kw = dict(defaults)
        for f in dataclasses.fields(cls):
            v = os.environ.get(prefix + f.name.upper())
            if v is None:
                continue
            if f.type in ("int", int):
                kw[f.name] = int(v)
            elif f.type in ("float", float):
                kw[f.name] = float(v)
            elif f.type in ("bool", bool):
                kw[f.name] = v.lower() in ("1", "true", "yes")
            elif f.name in ("byzantine_ranks", "straggler_ranks"):
                kw[f.name] = [int(x) for x in v.split(",") if x]
            else:
                kw[f.name] = v
        return cls(**kw).validate()

    def to_json(self) -> str:
        return json.dumps(dataclasses.asdict(self), sort_keys=True)
