"""Model-agnostic federated engine: any ``FlatNet`` (LeNet-5, ResNet-18, BERT-base, MLP) on the
same device-resident protocol as ``FusedEngine`` -- symmetric-heap upload buffers, epoch-tagged
P2P flags, the consensus/aggregation kernel, the host ledger re-executing every election.

A round is five launches: ``fed_plan_round``, the whole local-training pass as ONE captured
CUDA graph (forward, backward and optimizer of every mini-batch step -- all our kernels, no
host sync), ``fed_upload``, the committee's pull + validation of every candidate as a second
graph, ``fed_consensus_aggregate``.  Which graphs a rank replays is decided from the role
table it read back (104 bytes, pinned, non-blocking) at the end of the previous round -- no
device->host read inside a round.  (``capture()`` is optional: without it the same round runs
eagerly, kernel by kernel.)

Committee validation runs the model *directly on the trainers' HBM*: a candidate's ``Bound`` is a
set of tensor views over the peer-mapped upload buffers, so every GEMM of the forward pass
TMA-loads its weight tiles across NVLink -- the QueryAllUpdates all-gather (reference
C:299-311, M:196-217) never materialises.
"""
from __future__ import annotations

import struct
from typing import List, Optional

import torch
import torch.distributed as dist

from .._native import C, ledger as _ledger
from ..config import FLConfig
from ..data.synthetic import Shard
from ..models.nets import Bound, FlatNet
from ..parallel.layout import HeapLayout
from ..parallel.symm import SymmetricHeap
from .fused import ROLE_COMM, ROLE_TRAINER, FusedEngine, initial_roles


def vector_ranges(spec) -> torch.Tensor:
    """fp32 parts of an update that a forward pass reads from the master copy: every 1-D
    parameter (biases, norm scales / shifts, running statistics); matrices are consumed from
    the bf16 copy.  Coalesced {first float4, float4 count} pairs for ``fed_pull_candidates`` --
    for BERT-base this is 0.1 % of the 437 MB master.  int64 [n, 2] on the CPU."""
    runs = []
    for e in spec.entries:
        if len(e.shape) != 1:
            continue
        lo, hi = e.offset // 4, (e.offset + e.shape[0] + 3) // 4
        if runs and runs[-1][1] >= lo:
            runs[-1][1] = max(runs[-1][1], hi)
        else:
            runs.append([lo, hi])
    return torch.tensor([[lo, hi - lo] for lo, hi in runs], dtype=torch.int64).reshape(-1, 2)


class GenericFedEngine:
    read_state = FusedEngine.read_state
    drain_blocks = FusedEngine.drain_blocks
    read_stamps = FusedEngine.read_stamps

    def __init__(self, cfg: FLConfig, net: FlatNet, shard: Shard, *, rank: int = 0, world: int = 1,
                 device: int = 0, group=None):
        cfg.require_plain_fedavg("GenericFedEngine")
        assert cfg.clients == world and world <= 8
        self.cfg, self.net, self.rank, self.world, self.device = cfg, net, rank, world, device
        self.group = group
        torch.cuda.set_device(device)
        self.dev = torch.device("cuda", device)
        self.mod = C()
        # cfg.dtype "fp8": forward GEMMs of Linear / Conv2d run block-scaled fp8 (ops/mx8.py)
        from ..ops import nn as _nn
        _nn.set_precision("mx8" if cfg.dtype == "fp8" else "bf16")
        self.sz = sz = self.mod.struct_sizes()
        self.spec = net.spec
        P = self.n_params = net.spec.total
        B = cfg.batch_size
        self.S = (len(shard) // B) * B
        self.steps = (self.S // B) * cfg.local_epochs
        self.n_val = min(cfg.val_samples or len(shard), len(shard))
        self.layout = HeapLayout(P, cfg.ring_slots)
        self.heap = SymmetricHeap(self.layout.total_bytes, rank=rank, world=world, device=device,
                                  group=group, want_multicast=cfg.use_multicast)
        self.fed = self.layout.fed_dict(rank, world, self.heap.peer_ptrs, self.heap.mc_ptr)
        o, hv = self.layout.offsets, self.heap.view
        self.work_master = hv(o["work_master"], [P], torch.float32)
        self.work_shadow = hv(o["work_shadow"], [P], torch.bfloat16)
        self.global_master = hv(o["global"], [P], torch.float32)
        self.global_shadow = hv(o["global_shadow"], [P], torch.bfloat16)
        self.state_bytes = hv(o["state"], [sz["RoundState"]], torch.uint8)
        self.ring_bytes = hv(o["ring"], [cfg.ring_slots * sz["BlockRecord"]], torch.uint8)
        self.plan_bytes = hv(o["plan"], [sz["RoundPlan"]], torch.uint8)
        self.loss_sum = hv(o["plan"] + sz["plan_loss_sum_off"], [1], torch.float32)
        self.val_correct = hv(o["plan"] + sz["plan_correct_off"], [sz["kMaxRanks"]], torch.int32)
        self.opt_step_ptr = self.heap.local_ptr + o["plan"] + sz["plan_opt_step_off"]
        self.grad = torch.zeros(P, device=self.dev)
        self.m = torch.zeros(P, device=self.dev) if cfg.optimizer == "adam" else None
        self.v = torch.zeros(P, device=self.dev) if cfg.optimizer == "adam" else None

        init = torch.empty(P)
        net.init_(init, seed=cfg.seed + 1234)
        for t in (self.work_master, self.global_master):
            t.copy_(init)
        for t in (self.work_shadow, self.global_shadow):
            t.copy_(init.to(torch.bfloat16))
        self.bound = net.bind(self.work_master, self.work_shadow, self.grad)

        roles = initial_roles(cfg)
        st = self.mod.state_init_bytes(world, cfg.committee_size, cfg.aggregate_count, roles,
                                       cfg.needed_updates)
        self.state_bytes.copy_(torch.frombuffer(bytearray(st), dtype=torch.uint8))
        self.host_ledger = _ledger().Ledger(cfg.to_ledger_config(P))
        self.host_ledger.Bootstrap(roles)
        self.drained = 0

        self.x = net.preprocess(shard.x.to(self.dev))
        self.y = shard.y.to(self.dev, torch.int32)
        # big updates take the two-shot FedAvg (reduce a slice, publish it to every replica); small
        # ones the one-shot form.  (The fused engine also switches to two-shot from 8 ranks up; for
        # the generic engine that variant was not measured at 8 GPUs, so it stays opt-in: cfg.two_shot.)
        self.two_shot = cfg.two_shot if cfg.two_shot is not None else (P * 4 > (64 << 20) and world > 1)
        self.byz = 1 if rank in cfg.byzantine_ranks else 0
        self.straggle_us = cfg.straggler_delay_us if rank in cfg.straggler_ranks else 0
        self._peer_bounds = {}
        self._stage = None
        self._rounds = 0
        self.n_cand = world if cfg.solo else cfg.n_trainers      # candidates per round (fixed count)
        self.staged = bool(cfg.stage_candidates) and world > 1
        self.graph_train: Optional[torch.cuda.CUDAGraph] = None
        self.graph_val: Optional[torch.cuda.CUDAGraph] = None
        self.capture_error = ""
        self.stream = torch.cuda.Stream(device=self.dev)
        # role table cache: refreshed from the ledger page at the end of every round
        self._st_host = torch.empty(sz["RoundState"], dtype=torch.uint8).pin_memory()
        self._st_event = torch.cuda.Event()
        self._st = None
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize()

    # ------------------------------------------------------------------ pieces
    def peer_bound(self, t: int, parity: int) -> Bound:
        key = (t, parity)
        if key not in self._peer_bounds:
            o, P = self.layout.offsets, self.n_params
            master = self.heap.view(o[f"upload_master{parity}"], [P], torch.float32, rank=t)
            shadow = self.heap.view(o[f"upload_shadow{parity}"], [P], torch.bfloat16, rank=t)
            self._peer_bounds[key] = self.net.bind(master, shadow, None)
        return self._peer_bounds[key]

    def local_training(self):
        cfg, B = self.cfg, self.cfg.batch_size
        for i in range(self.steps):
            j = (i * B) % self.S
            loss = self.net.loss(self.bound, self.x[j:j + B], self.y[j:j + B])
            loss.backward()
            self.loss_sum += loss.detach() * B
            self.mod.optim_step(cfg.optimizer == "adam", self.work_master, self.grad,
                                self.work_shadow, self.m, self.v, cfg.learning_rate, 0.0, 0.9,
                                0.999, 1e-8, i + 1, self.opt_step_ptr, 0, True)

    def _vector_ranges(self) -> torch.Tensor:
        return vector_ranges(self.net.spec).to(self.dev)

    def _ensure_stage(self):
        if self._stage is None:
            P = self.n_params
            self._ranges = self._vector_ranges()
            self._stage = (torch.empty(self.world, P, device=self.dev, dtype=torch.bfloat16),
                           torch.empty(self.world, P, device=self.dev, dtype=torch.float32))
            self._stage_bounds = [self.net.bind(self._stage[1][z], self._stage[0][z], None)
                                  for z in range(self.world)]

    def validate_staged(self):
        """Committee: one P2P pass per candidate (bf16 weights + fp32 master) into local staging,
        started per candidate as soon as its trainer's flag is up (the kernel resolves the
        candidate -> trainer mapping from the ledger page), then the forward pass of every
        candidate slot out of local HBM.  No host-side knowledge of who the trainers are: the
        sequence is identical every round and therefore capturable."""
        xv, yv = self.x[: self.n_val], self.y[: self.n_val]
        self._ensure_stage()
        self.mod.fed_pull_candidates(self.fed, self._stage[0], self._stage[1],
                                     self._ranges if self._ranges.numel() else None)
        for z in range(self.n_cand):
            cnt = self.net.correct(self._stage_bounds[z], xv, yv)
            self.val_correct[z:z + 1].copy_(cnt)

    def validate(self, trainers: List[int], parity: int):
        xv, yv = self.x[: self.n_val], self.y[: self.n_val]
        if self.staged:
            self.validate_staged()
            return
        else:
            # direct: every GEMM of the forward pass TMA-loads its weight tiles from the peer
            self.mod.fed_wait_trained(self.fed)
            bounds = [self.peer_bound(t, parity) for t in trainers]
        for z, b in enumerate(bounds):
            cnt = self.net.correct(b, xv, yv)
            self.val_correct[z:z + 1].copy_(cnt)

    # ------------------------------------------------------------------ graphs
    def capture(self):
        """Warm up with one real (eager) round -- lazy kernel attribute setup, autograd graph
        buffers -- then capture the local-training pass and the staged validation pass.  Collective:
        every rank calls it.  Falls back to eager rounds if a capture fails (``capture_error``)."""
        self.run_round()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)
        if not self.cfg.cuda_graph:
            return
        # A rank that was committee in the warm-up round has never run the training body (and a
        # trainer never the validation forward): do both once, eagerly, on saved-and-restored
        # state, so that no first-use initialisation (lazy module loading, per-thread context
        # binding of autograd's worker, buffer caches) happens inside a capture.
        with torch.cuda.stream(self.stream):
            state = [t for t in (self.work_master, self.work_shadow, self.grad, self.m, self.v) if t is not None]
            keep = [t.clone() for t in state]
            plan = self.plan_bytes.clone()
            self.local_training()
            self.net.correct(self.bound, self.x[: self.n_val], self.y[: self.n_val])
            for t, k in zip(state, keep):
                t.copy_(k)
            self.plan_bytes.copy_(plan)
        torch.cuda.synchronize()
        del keep, plan
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream):
                self.local_training()
            self.graph_train = g
            if self.staged:      # (direct validation reads parity/trainer-dependent peer views: eager)
                gv = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gv, stream=self.stream):
                    self.validate_staged()
                self.graph_val = gv
        except Exception as e:  # noqa: BLE001
            self.graph_train = self.graph_val = None
            self.capture_error = repr(e)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)

    def _roles(self) -> dict:
        """Role table of the round about to start: read back at the end of the previous round."""
        if self._st is None:
            return self.read_state()
        self._st_event.synchronize()
        return self.read_state(self._st_host)

    # ------------------------------------------------------------------ one round
    def run_round(self) -> dict:
        m, cfg = self.mod, self.cfg
        # ring backpressure: drain the device BlockRecord ring before slots can be overwritten
        self._rounds += 1
        if self._rounds - self.drained >= max(cfg.ring_slots // 2, 1):
            errs = self.drain_blocks()
            if errs:
                raise RuntimeError(f"host/device ledgers disagree: {errs[:2]}")
        st = self._roles()
        role = st["roles"][self.rank]
        trainers = [r for r in range(self.world) if st["roles"][r] & ROLE_TRAINER]
        with torch.cuda.stream(self.stream):
            m.fed_plan_round(self.fed, [], self.steps, False)
            if role & ROLE_TRAINER:
                if self.graph_train is not None:
                    self.graph_train.replay()
                else:
                    self.local_training()
            m.fed_upload(self.fed, self.S, self.steps * cfg.batch_size, self.byz, cfg.byzantine_scale,
                         self.straggle_us)
            if role & ROLE_COMM:
                if self.graph_val is not None:
                    self.graph_val.replay()
                else:
                    self.validate(trainers, st["epoch"] & 1)
            m.fed_consensus_aggregate(self.fed, self.n_val, cfg.weight_by_score, self.two_shot,
                                      cfg.use_multicast and self.heap.has_multicast)
            # next round's role table: non-blocking readback of the ledger page
            self._st_host.copy_(self.state_bytes, non_blocking=True)
            self._st_event.record(self.stream)
            self._st = True
        torch.cuda.current_stream().wait_stream(self.stream)
        return st

    def evaluate(self, shard: Shard) -> float:
        x = self.net.preprocess(shard.x.to(self.dev))
        y = shard.y.to(self.dev, torch.int32)
        b = self.net.bind(self.global_master, self.global_shadow, None)
        return float(self.net.correct(b, x, y).item()) / len(shard)
