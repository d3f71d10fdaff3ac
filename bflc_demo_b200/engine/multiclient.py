"""Many clients on one GPU: the full committee protocol (committee scoring, median + top-K
filter, first-K admission, re-election) with C = 2..32 virtual clients sharing one device --
the reference's own 20 / 4 / 10 / 6 configuration runs here on a single B200.

Every buffer lives in local HBM (no symmetric heap, no P2P flags, no NCCL).  Its public surface
matches ``FusedEngine`` so callers can swap engines.

  round graph (one capture, no host sync inside; csrc/include/mc_round.h):
    k_mc_plan              QueryState for every client: trainer predicates, barrier words, Adam
                           step bases, committee list, simulated arrival order -> admitted set
    mlp_round  x C         local training, one persistent launch per client, predicated on that
                           client's trainer bit, launched one after another (a persistent
                           trainer's grid barrier needs all of its CTAs resident at once)
    k_mc_byzantine         fault injection: update := global - s * (trained - global)
    [fp8] quantize x C     each client's candidate blob from its trained master
    mc_val                 every committee member scores every admitted candidate on its own
                           n_val_c rows: ONE launch over (m-tile, candidate, member)
    k_mc_consensus         scores, run_consensus<32>, ledger page, block record
    k_mc_fedavg            deterministic FedAvg into the global model and every client
    [fp8] quantize + k_mc_bcast   the new global blob into every client's training copy

Every trainer trains, also those that will not be admitted (the reference rejects at upload).

Clients may hold shards of different sizes (and label mixes).  Client c with rows_c rows trains
S_c = (rows_c // B) * B samples in steps_c = S_c / B * local_epochs steps, validates as a committee
member on n_val_c = min(val_samples or rows_c, rows_c) rows of its own shard and reports
n_samples = S_c, so FedAvg weights the selected clients by their sample counts -- the rule
``FusedEngine`` applies per rank.  These constants live in the device-resident ``McClients``.

Against client drift under skewed data (DESIGN.md, "FedProx and server optimizers"):
``cfg.prox_mu`` > 0 adds the FedProx term mu/2 ||w - w_global||^2 to every client's local loss (the
anchor is ``global_master``, which holds the round-start model for the whole training phase), and
``cfg.server_optimizer`` (momentum | adam | yogi) turns the FedAvg step into a server optimizer
step on the pseudo-gradient average - global, with its state in ``server_m`` / ``server_v``.  The
committee, the election, the FedAvg weights and the host ledger are the same in every setting.
"""
from __future__ import annotations

import struct
from typing import Dict, List, Optional, Sequence

import torch

from .._native import C, ledger as _ledger
from ..config import FLConfig
from ..data.synthetic import Shard
from ..models.mlp import FlatMLP, mlp_spec, sf_bytes
from ..ops import gemm as G
from .fused import ROLE_COMM, ROLE_TRAINER, initial_roles

MAX_CLIENTS = 32

# McState: epoch, n_clients, n_comm, n_aggregate, n_needed, seed, straggler_mask, blocks_appended,
# role[32], last_median[32], admitted_mask, selected_mask, global_loss, pad, model_digest
_MC_STATE = struct.Struct("<8I32I32f2IfIQ")
# McBlockRecord: epoch, n_clients, n_comm, n_aggregate, role_before[32], role_after[32],
# score_rows[32][32], scored_mask[32], median[32], n_samples[32], avg_cost[32], weight[32],
# admitted_mask, selected_mask, global_loss, weight_by_score, model_digest, seq, pad
_MC_REC = struct.Struct("<4I32I32I1024f32I32f32I32f32f2IfIQ2I")


class MultiClientEngine:
    def __init__(self, cfg: FLConfig, shards: Sequence[Shard], device: int = 0):
        cfg.validate()
        n = cfg.clients
        if not (2 <= n <= MAX_CLIENTS) or cfg.solo:
            raise ValueError(f"MultiClientEngine runs 2..{MAX_CLIENTS} clients with a committee (solo=False)")
        if len(shards) != n:
            raise ValueError(f"need one shard per client ({n}), got {len(shards)}")
        self.cfg, self.device = cfg, device
        torch.cuda.set_device(device)
        self.dev = torch.device("cuda", device)
        self.mod = m = C()
        sz = m.struct_sizes()
        self.sz = sz
        assert sz["McState"] == _MC_STATE.size and sz["McBlockRecord"] == _MC_REC.size, \
            "multi-client struct layout changed: update _MC_STATE / _MC_REC"

        n_classes = shards[0].n_classes
        B = cfg.batch_size
        self.fp8 = cfg.dtype == "fp8"
        rows_c = [len(s) for s in shards]
        for c, s in enumerate(shards):
            if s.n_classes != n_classes:
                raise ValueError(f"client {c} has {s.n_classes} classes, client 0 has {n_classes}: "
                                 "every shard must have the same class count")
            if rows_c[c] < B:
                raise ValueError(f"client {c} holds {rows_c[c]} rows, fewer than one batch ({B})")
            if self.fp8 and rows_c[c] % 128:
                raise ValueError(f"dtype='fp8' needs shard rows % 128 == 0; client {c} holds {rows_c[c]}")
        self.in_dim = shards[0].x.reshape(rows_c[0], -1).shape[1]
        if any(s.x.reshape(len(s), -1).shape[1] != self.in_dim for s in shards):
            raise ValueError("every client shard must have the same feature size")
        self.spec = mlp_spec(self.in_dim, cfg.hidden, n_classes)
        self.n_params = P = self.spec.total
        self.n_classes = n_classes
        # per-client shard constants (the same rule as FusedEngine applies per rank)
        self.rows_per_client = rows_c
        self.samples_per_client = [(r // B) * B for r in rows_c]
        self.steps_per_client = [(S // B) * cfg.local_epochs for S in self.samples_per_client]
        self.n_val_per_client = [min(cfg.val_samples or r, r) for r in rows_c]
        # equal shards: the scalars of a uniform engine; unequal shards: None (use the lists)
        def uniform(v):
            return v[0] if all(x == v[0] for x in v) else None
        self.rows = uniform(self.rows_per_client)
        self.S = uniform(self.samples_per_client)
        self.steps = uniform(self.steps_per_client)
        self.n_val = uniform(self.n_val_per_client)
        if cfg.dtype not in ("bf16", "fp8"):
            raise ValueError("MultiClientEngine: dtype must be bf16 or fp8")
        if not (cfg.hidden == 256 and n_classes <= 64 and self.in_dim % 16 == 0):
            raise ValueError("MultiClientEngine runs the flagship MLP: hidden == 256, <= 64 classes, "
                             "in_dim % 16 == 0")
        if self.fp8 and B % 128:
            raise ValueError("dtype='fp8' needs batch % 128 == 0")

        # ---- per-client model state: [C, P] master / shadow / grad, own Adam moments ---------
        dev = self.dev
        self.master = torch.zeros(n, P, device=dev, dtype=torch.float32)
        self.shadow = torch.zeros(n, P, device=dev, dtype=torch.bfloat16)
        self.grad = torch.zeros(n, P, device=dev, dtype=torch.float32)
        self.global_master = torch.zeros(P, device=dev, dtype=torch.float32)
        self.global_shadow = torch.zeros(P, device=dev, dtype=torch.bfloat16)
        init = torch.empty(P, dtype=torch.float32)
        self.spec.init_(init, seed=cfg.seed + 1234)
        for t in (self.global_master, self.master):
            t.copy_(init.to(dev).expand_as(t))
        for t in (self.global_shadow, self.shadow):
            t.copy_(init.to(dev, torch.bfloat16).expand_as(t))

        # ---- ledger page, plan, block ring ----------------------------------------------------
        self.state_bytes = torch.zeros(sz["McState"], device=dev, dtype=torch.uint8)
        self.plan_bytes = torch.zeros(sz["McPlan"], device=dev, dtype=torch.uint8)
        self.ring_bytes = torch.zeros(cfg.ring_slots * sz["McBlockRecord"], device=dev, dtype=torch.uint8)
        self.plan_ptr = pp = self.plan_bytes.data_ptr()
        roles = initial_roles(cfg)
        strag = sum(1 << r for r in cfg.straggler_ranks if 0 <= r < n)
        st = m.mc_state_init_bytes(n, cfg.committee_size, cfg.aggregate_count, cfg.needed_updates,
                                   cfg.seed, strag, roles)
        self.state_bytes.copy_(torch.frombuffer(bytearray(st), dtype=torch.uint8))
        self.host_ledger = _ledger().Ledger(cfg.to_ledger_config(P))
        self.host_ledger.Bootstrap(roles)
        self.drained = 0

        def plan_view(key, count, dtype):
            off = sz[key]
            nbytes = count * torch.empty(0, dtype=dtype).element_size()
            return self.plan_bytes[off:off + nbytes].view(dtype)

        self.loss_sum = plan_view("mc_plan_loss_sum_off", MAX_CLIENTS, torch.float32)
        self.train_correct = plan_view("mc_plan_train_correct_off", MAX_CLIENTS, torch.int32)
        self.correct = plan_view("mc_plan_correct_off", MAX_CLIENTS * MAX_CLIENTS, torch.int32).view(
            MAX_CLIENTS, MAX_CLIENTS)

        # ---- server optimizer state: m = 0, v = tau^2 at genesis (Reddi et al., Algorithm 2) ---
        so = cfg.server_optimizer
        self.server_m = torch.zeros(P, device=dev, dtype=torch.float32) if so != "none" else None
        self.server_v = (torch.full((P,), cfg.server_tau * cfg.server_tau, device=dev, dtype=torch.float32)
                         if so in ("adam", "yogi") else None)
        self.server_kw = dict(server_optimizer=so, lr=cfg.server_lr, beta1=cfg.server_beta1,
                              beta2=cfg.server_beta2, tau=cfg.server_tau,
                              m=self.server_m.data_ptr() if self.server_m is not None else 0,
                              v=self.server_v.data_ptr() if self.server_v is not None else 0)

        # ---- one persistent trainer per client (own barrier word, step base, Adam moments);
        #      FedProx anchors every client to the round-start global model
        self.trainers: List[FlatMLP] = []
        for c in range(n):
            tr = FlatMLP(self.spec, self.master[c], self.shadow[c], self.grad[c], B,
                         optimizer=cfg.optimizer, lr=cfg.learning_rate,
                         loss_sum=self.loss_sum[c:c + 1], correct=self.train_correct[c:c + 1],
                         step_dev_ptr=pp + sz["mc_plan_opt_step_off"] + 4 * c, fp8=self.fp8,
                         prox_mu=cfg.prox_mu, prox_anchor=self.global_master if cfg.prox_mu > 0 else None)
            if not tr.fused_ok(self.steps_per_client[c]):
                raise ValueError("shape outside the persistent trainer's limits")
            self.trainers.append(tr)
        self.ql = m.mx8_mlp_layout(self.in_dim, cfg.hidden) if self.fp8 else None
        self.byz_ids = sorted(r for r in set(cfg.byzantine_ranks) if 0 <= r < n)

        # ---- resident inputs, converted once: one ragged allocation per tensor, client c's rows
        #      at a 128-row aligned offset, exposed as per-client views x_bf[c], y[c], x_q[c], x_sf[c]
        D = self.in_dim
        row_off, sf_off, r0, f0 = [], [], 0, 0
        for r in rows_c:
            row_off.append(r0)
            sf_off.append(f0)
            r0 += -(-r // 128) * 128
            f0 += sf_bytes(r, D)
        x_bf_all = torch.empty(r0, D, device=dev, dtype=torch.bfloat16)
        y_all = torch.zeros(r0, device=dev, dtype=torch.int32)
        x_q_all = torch.zeros(r0, D, device=dev, dtype=torch.uint8) if self.fp8 else None
        x_sf_all = torch.full((f0,), 127, device=dev, dtype=torch.uint8) if self.fp8 else None
        self.x_bf = [x_bf_all[o:o + r] for o, r in zip(row_off, rows_c)]
        self.y = [y_all[o:o + r] for o, r in zip(row_off, rows_c)]
        self.x_q = [x_q_all[o:o + r] for o, r in zip(row_off, rows_c)] if self.fp8 else None
        self.x_sf = [x_sf_all[o:o + sf_bytes(r, D)] for o, r in zip(sf_off, rows_c)] if self.fp8 else None
        for c, s in enumerate(shards):
            xu = s.x.reshape(rows_c[c], -1).to(dev, torch.uint8).contiguous()
            m.prep_inputs(xu, self.x_bf[c], self.x_q[c] if self.fp8 else None,
                          self.x_sf[c] if self.fp8 else None, 1.0 / 255.0)
            self.y[c].copy_(s.y.to(torch.int32))

        blobs = [t.work_q.data_ptr() for t in self.trainers] if self.fp8 else []
        self.clients_dev = torch.frombuffer(bytearray(m.mc_clients_bytes(
            [self.master[c].data_ptr() for c in range(n)], [self.shadow[c].data_ptr() for c in range(n)],
            blobs, [self.y[c].data_ptr() for c in range(n)],
            [self.x_sf[c].data_ptr() for c in range(n)] if self.fp8 else [],
            self.samples_per_client, self.steps_per_client, self.n_val_per_client, B)),
            dtype=torch.uint8).to(dev)
        self.args = dict(st=self.state_bytes.data_ptr(), plan=pp, ring=self.ring_bytes.data_ptr(),
                         ring_slots=cfg.ring_slots, clients=self.clients_dev.data_ptr(),
                         global_master=self.global_master.data_ptr(),
                         global_shadow=self.global_shadow.data_ptr(), n_params=P)

        # ---- validation tensor maps: x of every client (its first n_val_c rows), [layer][client]
        #      weights read in place (bf16 work shadow, or the client's fp8 blob) --------------
        K = MAX_CLIENTS
        CTM = sz["CUtensorMap"]
        xm, wm = bytearray(K * CTM), bytearray(2 * K * CTM)
        e1, e2 = self.spec.by_name["w1"], self.spec.by_name["w2"]
        for c in range(n):
            xsrc = self.x_q[c] if self.fp8 else self.x_bf[c]
            xm[c * CTM:(c + 1) * CTM] = m.operand_map(xsrc.data_ptr(), D, self.n_val_per_client[c], D,
                                                      self.fp8, 128)
            if self.fp8:
                base = self.trainers[c].work_q.data_ptr()
                w1 = m.gemm_b_map(base + self.ql["w1q"], e1.shape[0], D, D, False, True, G.EPI_GENERIC, 256)
                w2 = m.gemm_b_map(base + self.ql["w2q"], 64, cfg.hidden, cfg.hidden, False, True, G.EPI_ARGMAX, 64)
            else:
                base = self.shadow[c].data_ptr()
                w1 = m.gemm_b_map(base + e1.offset * 2, e1.shape[0], D, D, False, False, G.EPI_GENERIC, 256)
                w2 = m.gemm_b_map(base + e2.offset * 2, e2.shape[0], e2.shape[1], e2.shape[1], False, False,
                                  G.EPI_ARGMAX, 64)
            wm[c * CTM:(c + 1) * CTM] = w1
            wm[(K + c) * CTM:(K + c + 1) * CTM] = w2
        self.x_maps = torch.frombuffer(xm, dtype=torch.uint8).to(dev)
        self.w_maps = torch.frombuffer(wm, dtype=torch.uint8).to(dev)
        self.max_cand = min(cfg.needed_updates, cfg.n_trainers)

        # fp8: every client's training copy starts as the quantised genesis model
        if self.fp8:
            self.global_blob = torch.zeros(self.ql["total"], device=dev, dtype=torch.uint8)
            self._broadcast_global_blob()

        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self._rounds = 0
        self.launches_per_round = 0
        self.stream = torch.cuda.Stream(device=dev)
        torch.cuda.synchronize()

    # ------------------------------------------------------------------ one round, by phase
    def _broadcast_global_blob(self):
        self.trainers[0].quantize_weights(self.global_master, self.global_blob)
        self.mod.mc_broadcast_blob(self.args, self.global_blob, self.cfg.clients)

    def phase_train(self):
        """Plan + local training of every trainer (+ Byzantine injection, + candidate blobs)."""
        m, cfg, sz = self.mod, self.cfg, self.sz
        m.mc_plan_round(self.args)
        for c, tr in enumerate(self.trainers):
            m.set_predicate(self.plan_ptr + sz["mc_plan_is_trainer_off"] + 4 * c)
            tr.train_epoch_fused(self.x_bf[c], self.y[c], self.steps_per_client[c],
                                 self.plan_ptr + sz["mc_plan_barrier_off"] + 4 * c,
                                 x_q=self.x_q[c] if self.fp8 else None,
                                 x_sf=self.x_sf[c] if self.fp8 else None)
        m.set_predicate(0)
        m.mc_byzantine(self.args, self.byz_ids, cfg.byzantine_scale)
        if self.fp8:
            # candidate = the trained (or Byzantine) master, quantised; the trainer's optimizer
            # epilogue refreshes only the weight matrices of its blob, not the biases
            for tr in self.trainers:
                tr.quantize_weights()

    def phase_validate(self):
        """Committee validation: correct[member][candidate] in one launch."""
        m, sz = self.mod, self.sz
        e = self.spec.by_name
        m.mc_val(self.plan_ptr, self.plan_ptr + sz["mc_plan_correct_off"], self.x_maps, self.w_maps,
                 self.clients_dev.data_ptr(), e["b1"].offset, e["b2"].offset, max(self.n_val_per_client),
                 self.in_dim, self.cfg.hidden, self.n_classes, self.max_cand, self.cfg.committee_size, self.fp8)

    def phase_aggregate(self):
        """Consensus, ledger page, block record, FedAvg (+ server optimizer step) into the global
        model and every client."""
        m, cfg = self.mod, self.cfg
        m.mc_consensus(self.args, cfg.weight_by_score)
        self.fedavg()
        if self.fp8:
            self._broadcast_global_blob()

    def fedavg(self):
        """The FedAvg kernel alone, with this engine's server optimizer."""
        self.mod.mc_fedavg(self.args, self.cfg.clients, **self.server_kw)

    def _enqueue_round(self):
        n0 = self.mod.launch_count()
        self.phase_train()
        self.phase_validate()
        self.phase_aggregate()
        self.launches_per_round = int(self.mod.launch_count() - n0)

    def capture(self):
        """One eager round (warm-up: lazy kernel setup), then capture the round graph."""
        with torch.cuda.stream(self.stream):
            self._enqueue_round()
        self.stream.synchronize()
        self._rounds += 1
        if not self.cfg.cuda_graph:
            return
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self.stream):
            self._enqueue_round()
        self.graph = g

    def run_round(self):
        # the ring holds ring_slots records: drain into the host ledger before any is overwritten
        self._rounds += 1
        if self._rounds - self.drained >= max(self.cfg.ring_slots // 2, 1):
            errs = self.drain_blocks()
            if errs:
                raise RuntimeError(f"host/device ledgers disagree: {errs[:2]}")
        with torch.cuda.stream(self.stream):
            if self.graph is not None:
                self.graph.replay()
            else:
                self._enqueue_round()

    # ------------------------------------------------------------------ host views
    def read_state(self) -> dict:
        torch.cuda.synchronize()
        f = _MC_STATE.unpack(bytes(self.state_bytes.cpu().numpy()))
        n = self.cfg.clients
        return dict(epoch=f[0], roles=list(f[8:8 + n]), median=list(f[40:40 + n]), admitted_mask=f[72],
                    selected_mask=f[73], global_loss=f[74], model_digest=f[76])

    def drain_blocks(self) -> List[str]:
        """Finished McBlockRecords -> host C++ ledger, which re-executes every election.  The
        device's FedAvg weight of every selected client must equal the host block's bit for bit
        (both sides compute it in double in the shared run_consensus).
        Returns the mismatches ([] = device and host agree)."""
        torch.cuda.synchronize()
        st = self.read_state()
        ring = bytes(self.ring_bytes.cpu().numpy())
        rs, n, K = _MC_REC.size, self.cfg.clients, MAX_CLIENTS
        errs: List[str] = []
        dev_weights: List[tuple] = []          # (epoch, record weight[0..n)) of appended blocks
        while self.drained < st["epoch"]:
            e = self.drained
            f = _MC_REC.unpack_from(ring, (e % self.cfg.ring_slots) * rs)
            p = 4
            role_before = f[p:p + n]; p += K
            role_after = f[p:p + n]; p += K
            rows = [list(f[p + K * c:p + K * c + n]) for c in range(n)]; p += K * K
            scored = f[p:p + n]; p += K
            p += K                                   # median
            n_samples = f[p:p + n]; p += K
            avg_cost = f[p:p + n]; p += K
            weight = f[p:p + n]; p += K
            adm, sel, gl, wbs, digest, seq = f[p:p + 6]
            if f[0] != e or seq != e + 1:
                errs.append(f"ring slot for epoch {e} holds epoch {f[0]} seq {seq}")
                break
            msg = self.host_ledger.AppendDeviceRound(dict(
                epoch=e, role_before=list(role_before), role_after=list(role_after), score_rows=rows,
                scored_mask=list(scored), n_samples=list(n_samples), avg_cost=list(avg_cost),
                admitted_mask=adm, selected_mask=sel, global_loss=gl, model_digest=digest,
                weight_by_score=wbs))
            if msg:
                errs.append(f"epoch {e}: {msg}")
                break
            dev_weights.append((e, weight))
            self.drained += 1
        if dev_weights:
            blocks = self.host_ledger.blocks()[-len(dev_weights):]
            for (e, weight), blk in zip(dev_weights, blocks):
                if blk["epoch"] != e:
                    errs.append(f"epoch {e}: host block holds epoch {blk['epoch']}")
                    continue
                for t, w in zip(blk["selected"], blk["weight"]):
                    if weight[t] != w:
                        errs.append(f"epoch {e}: FedAvg weight of client {t}: device {weight[t]!r} "
                                    f"host {w!r}")
        return errs

    def committee(self) -> List[int]:
        return [c for c, r in enumerate(self.read_state()["roles"]) if r & ROLE_COMM]

    def trainers_now(self) -> List[int]:
        return [c for c, r in enumerate(self.read_state()["roles"]) if r & ROLE_TRAINER]

    def global_model(self) -> Dict[str, torch.Tensor]:
        return {k: v.clone() for k, v in self.spec.views(self.global_master).items()}

    def evaluate(self, shard: Shard) -> float:
        """Sponsor-style test accuracy of the current global model (M:285-306)."""
        x = shard.x.reshape(len(shard), -1).to(self.dev)
        xb = torch.empty(x.shape, device=self.dev, dtype=torch.bfloat16)
        self.mod.prep_inputs(x.contiguous(), xb, None, None, 1.0 / 255.0)
        cnt = self.trainers[0].accuracy_counts(xb, shard.y.to(self.dev, torch.int32),
                                                shadow=self.global_shadow, master=self.global_master)
        return float(cnt.item()) / len(shard)
