"""OUR NCCL + cuBLAS baseline of the reference algorithm (NOT a reference-published build:
iammcy/BFLC-demo ships no GPU code and cannot be built offline -- SURVEY.md 0.3, BASELINE.md).

Same protocol, same model, same data as ``FusedEngine``, built the conventional way and tuned
the way a competent PyTorch user would (SURVEY.md 7.5.8) -- this is the number the fused engine
is compared against in ``bench.py``'s ``vs_baseline``:

  * local training: cuBLASLt GEMMs with fused bias / bias+ReLU epilogues
    (``torch._addmm_activation``), persistent bf16 shadow weights refreshed by one multi-tensor
    copy per step, ``log_softmax``-based cross-entropy, multi-tensor SGD or ``_fused_adam_``;
  * the exchanges are NCCL collectives on pre-allocated flat buffers: one ``all_gather`` of
    [weights | n_samples | avg_cost] and one ``all_gather`` of the score rows;
  * the election (true median -> stable top-K -> sample weights -> re-election) runs ON THE
    DEVICE with torch ops, so nothing blocks in the middle of a round;
  * the WHOLE round -- training, both collectives, validation, election, FedAvg (a single GEMV)
    -- is ONE captured CUDA graph per role (trainer / committee / solo); the host only picks the
    graph, from the role table it read back (16 bytes, pinned, non-blocking) at the end of the
    previous round.

What it cannot avoid is what the fused engine is built to remove: collectives as separate
kernels behind a host-chosen graph, weights crossing NVLink as fp32 all-gathers to every rank,
~10^2 small kernels per round.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.distributed as dist

from ..config import FLConfig
from ..data.synthetic import Shard
from ..models.mlp import mlp_spec
from .fused import ROLE_COMM, ROLE_TRAINER, initial_roles


class NcclBaselineEngine:
    def __init__(self, cfg: FLConfig, shard: Shard, *, rank: int = 0, world: int = 1,
                 device: int = 0, group=None, broadcast: bool = False):
        cfg.require_plain_fedavg("NcclBaselineEngine")
        self.cfg, self.rank, self.world, self.group = cfg, rank, world, group
        self.dev = torch.device("cuda", device)
        torch.cuda.set_device(device)
        self.broadcast = broadcast
        x0 = shard.x.reshape(len(shard), -1)
        self.in_dim = x0.shape[1]
        self.spec = mlp_spec(self.in_dim, cfg.hidden, shard.n_classes)
        P = self.P = self.spec.total
        B = cfg.batch_size
        self.S = (len(shard) // B) * B
        self.steps = (self.S // B) * cfg.local_epochs
        self.n_val = min(cfg.val_samples or len(shard), len(shard))
        init = torch.empty(P)
        self.spec.init_(init, seed=cfg.seed + 1234)
        self.global_w = init.to(self.dev)
        # upload record of this rank: [weights (P) | n_samples | avg_cost | pad] in ONE buffer so
        # a single all_gather moves everything the aggregation needs
        self.rec = P + 8
        self.mine = torch.zeros(self.rec, device=self.dev)
        self.work = self.mine[:P]
        self.work.copy_(self.global_w)
        self.wv = self.spec.views(self.work)
        self.names = ("w1", "b1", "w2", "b2")
        self.params = [self.wv[k] for k in self.names]
        self.shadow = torch.zeros(P, device=self.dev, dtype=torch.bfloat16)
        self.sv = self.spec.views(self.shadow)
        self.shadows = [self.sv[k] for k in self.names]
        self.adam = cfg.optimizer == "adam"
        if self.adam:
            self.m = [torch.zeros_like(p) for p in self.params]
            self.v = [torch.zeros_like(p) for p in self.params]
            self.t = [torch.zeros((), device=self.dev) for _ in self.params]
        self.all_rec = torch.zeros(world, self.rec, device=self.dev)
        self.all_scores = torch.zeros(world, world, device=self.dev)
        self.my_scores = torch.zeros(world, device=self.dev)
        self.roles_dev = torch.tensor(initial_roles(cfg), device=self.dev, dtype=torch.int32)
        self.roles: List[int] = initial_roles(cfg)
        self.epoch = 0
        self.global_loss = 0.0
        self.gl_dev = torch.zeros(1, device=self.dev)
        self.host_x = x0.contiguous().pin_memory()
        self.host_y = shard.y.to(torch.int64).contiguous().pin_memory()
        self.x_u8 = self.host_x.to(self.dev)
        self.y = self.host_y.to(self.dev)
        self.x_bf = torch.empty(len(shard), self.in_dim, device=self.dev, dtype=torch.bfloat16)
        self.loss_acc = torch.zeros(1, device=self.dev)
        self.minus_one = torch.full((B, 1), -1.0, device=self.dev)
        self.ar = torch.arange(world, device=self.dev)
        self.stream = torch.cuda.Stream(device=self.dev)
        self.graphs = {}
        # end-of-round readback: roles (int32[world]) + global loss, pinned, non-blocking
        self.out_host = torch.zeros(world + 1, dtype=torch.float32).pin_memory()
        self.out_dev = torch.zeros(world + 1, device=self.dev)
        self.byz = rank in cfg.byzantine_ranks
        try:    # cuBLAS writes fp32 straight out of a bf16 GEMM when torch exposes out_dtype
            a = torch.zeros(8, 8, device=self.dev, dtype=torch.bfloat16)
            torch.mm(a, a, out_dtype=torch.float32)
            self._mm32 = lambda a, b: torch.mm(a, b, out_dtype=torch.float32)
        except Exception:  # noqa: BLE001
            self._mm32 = lambda a, b: (a @ b).float()

    # ---------------------------------------------------------------- local work
    def _train_pass(self):
        cfg = self.cfg
        B, lr = cfg.batch_size, cfg.learning_rate
        w, s = self.wv, self.sv
        self.work.copy_(self.global_w)
        torch._foreach_copy_(self.shadows, self.params)
        self.loss_acc.zero_()
        for i in range(self.steps):
            x = self.x_bf[i * B:(i + 1) * B]
            y = self.y[i * B:(i + 1) * B]
            # cuBLASLt: bias + ReLU in the GEMM epilogue
            h = torch._addmm_activation(s["b1"], x, s["w1"].t(), use_gelu=False)
            logits = torch.addmm(s["b2"], h, s["w2"].t())
            logp = torch.log_softmax(logits, 1, dtype=torch.float32)       # cast fused into the softmax
            self.loss_acc += torch.nn.functional.nll_loss(logp, y, reduction="sum")
            p = torch.exp(logp)
            p.scatter_add_(1, y[:, None], self.minus_one)
            dlf = p * (1.0 / B)
            dl = dlf.to(torch.bfloat16)
            gw2 = self._mm32(dl.t(), h)                                    # bf16 x bf16 -> fp32 out
            gb2 = dlf.sum(0)
            dh = torch.ops.aten.threshold_backward(dl @ s["w2"], h, 0)     # fused relu'
            gw1 = self._mm32(dh.t(), x)
            gb1 = dh.sum(0, dtype=torch.float32)
            grads = [gw1, gb1, gw2, gb2]
            if self.adam:
                torch._foreach_add_(self.t, 1.0)
                torch._fused_adam_(self.params, grads, self.m, self.v, [], self.t, lr=lr, beta1=0.9,
                                   beta2=0.999, weight_decay=0.0, eps=1e-8, amsgrad=False, maximize=False)
            else:
                torch._foreach_add_(self.params, grads, alpha=-lr)
            torch._foreach_copy_(self.shadows, self.params)
        if self.byz:
            self.work.copy_(self.global_w - self.cfg.byzantine_scale * (self.work - self.global_w))
        self.mine[self.P:self.P + 1].fill_(float(self.S))
        self.mine[self.P + 1:self.P + 2] = self.loss_acc / float(self.steps * B)

    def _val_pass(self):
        """Score every CANDIDATE (= this round's trainers; their ranks are data, their count is
        fixed) on this committee member's shard: two batched cuBLAS GEMMs."""
        xv = self.x_bf[: self.n_val]
        yv = self.y[: self.n_val]
        nc = self.cfg.n_trainers
        tr = ((self.roles_dev & ROLE_TRAINER) > 0).int()
        cand = torch.sort(tr, descending=True, stable=True).indices[:nc]     # trainer ranks, ascending
        W = self.all_rec.index_select(0, cand)[:, : self.P].to(torch.bfloat16)
        e = self.spec.by_name

        def part(name):
            en = e[name]
            return W[:, en.offset:en.offset + en.numel].reshape(nc, *en.shape)
        w1, b1, w2, b2 = part("w1"), part("b1"), part("w2"), part("b2")
        h = torch.relu(torch.baddbmm(b1[:, None, :], xv[None].expand(nc, -1, -1), w1.transpose(1, 2)))
        logits = torch.baddbmm(b2[:, None, :], h, w2.transpose(1, 2))
        self.my_scores.zero_()
        self.my_scores.index_copy_(0, cand, (logits.argmax(2) == yv[None]).float().mean(1))

    def _elect_and_apply(self):
        """Aggregate (C:349-456) with torch ops on the device: true median over the committee rows,
        stable descending sort (ties -> ascending rank), top-K sample-weighted FedAvg as one GEMV,
        re-election with refill from the outgoing committee."""
        cfg, n = self.cfg, self.world
        roles = self.roles_dev
        comm = (roles & ROLE_COMM) > 0
        tr = (roles & ROLE_TRAINER) > 0
        k = comm.sum()
        S = torch.where(comm[:, None], self.all_scores, torch.full_like(self.all_scores, float("inf")))
        srt = S.sort(0).values
        lo = srt.gather(0, ((k - 1) // 2).clamp(min=0).expand(1, n)).squeeze(0)
        hi = srt.gather(0, (k // 2).expand(1, n)).squeeze(0)
        med = torch.where(tr, 0.5 * (lo + hi), torch.full_like(lo, float("-inf")))
        order = torch.sort(med, descending=True, stable=True).indices
        pos = torch.empty_like(order)
        pos[order] = self.ar
        n_tr = tr.sum()
        n_sel = torch.clamp(n_tr, max=cfg.aggregate_count)
        sel = (pos < n_sel) & tr
        ns = self.all_rec[:, self.P]
        w = ns * sel
        if cfg.weight_by_score:
            w = w * torch.where(sel, med, torch.zeros_like(med))
        wsum = w.sum()
        w = torch.where(wsum > 0, w / wsum.clamp(min=1e-30), sel.float() / n_sel.clamp(min=1))
        has = n_sel > 0
        new_global = torch.mv(self.all_rec[:, : self.P].t(), w)
        self.global_w.copy_(torch.where(has, new_global, self.global_w))
        self.gl_dev.copy_(((self.all_rec[:, self.P + 1] * sel).sum() / n_sel.clamp(min=1)).reshape(1))
        # re-election
        solo = (comm & tr).any()
        elected = (pos < cfg.committee_size) & tr
        need = cfg.committee_size - elected.sum()
        refill_pool = comm & ~elected
        refill = refill_pool & (torch.cumsum(refill_pool.int(), 0) <= need)
        new_roles = torch.where(elected | refill, ROLE_COMM, ROLE_TRAINER).to(torch.int32)
        self.roles_dev.copy_(torch.where(solo, roles, new_roles))
        if self.broadcast and n > 1:          # the literal BASELINE.json loop: rank 0 publishes
            dist.broadcast(self.global_w, src=0, group=self.group)
        self.out_dev[:n].copy_(self.roles_dev.float())
        self.out_dev[n:].copy_(self.gl_dev)

    def _round_body(self, train: bool, validate: bool):
        n = self.world
        self.x_bf.copy_(self.x_u8)
        self.x_bf.mul_(1.0 / 255.0)
        if train:
            self._train_pass()
        if n > 1:
            dist.all_gather_into_tensor(self.all_rec.view(-1), self.mine, group=self.group)
        else:
            self.all_rec[0].copy_(self.mine)
        if validate:
            self._val_pass()
        if n > 1:
            dist.all_gather_into_tensor(self.all_scores.view(-1), self.my_scores, group=self.group)
        else:
            self.all_scores[0].copy_(self.my_scores)
        self._elect_and_apply()

    def capture(self):
        """Warm up every role's round once eagerly (lazy cuBLAS / NCCL setup; collective, every
        rank runs the same sequence), restore the genesis state, then capture one graph per role."""
        snap = (self.global_w.clone(), self.roles_dev.clone())
        combos = [(True, True)] if self.cfg.solo else [(True, False), (False, True)]
        with torch.cuda.stream(self.stream):
            for tv in combos:
                self._round_body(*tv)
        self.stream.synchronize()
        if self.cfg.cuda_graph:
            for tv in combos:
                g = torch.cuda.CUDAGraph()
                try:
                    with torch.cuda.graph(g, stream=self.stream):
                        self._round_body(*tv)
                    self.graphs[tv] = g
                except Exception as e:  # noqa: BLE001  (NCCL capture unsupported: run eagerly)
                    self.graphs = {}
                    self.capture_error = repr(e)
                    break
        self.global_w.copy_(snap[0])
        self.roles_dev.copy_(snap[1])
        self.work.copy_(self.global_w)
        if self.adam:
            torch._foreach_zero_(self.m + self.v + self.t)
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- one round
    def run_round(self) -> dict:
        role = self.roles[self.rank]
        tv = (bool(role & ROLE_TRAINER), bool(role & ROLE_COMM))
        with torch.cuda.stream(self.stream):
            g = self.graphs.get(tv)
            if g is not None:
                g.replay()
            else:
                self._round_body(*tv)
            self.out_host.copy_(self.out_dev, non_blocking=True)
        # the host needs the new role table to pick the next round's graph
        self.stream.synchronize()
        n = self.world
        self.roles = [int(v) for v in self.out_host[:n].tolist()]
        self.global_loss = float(self.out_host[n])
        self.epoch += 1
        return dict(epoch=self.epoch, roles=list(self.roles), global_loss=self.global_loss)

    def run_round_e2e(self, host_x=None, host_y=None) -> dict:
        hx = self.host_x if host_x is None else host_x
        hy = self.host_y if host_y is None else host_y
        with torch.cuda.stream(self.stream):
            self.x_u8.copy_(hx, non_blocking=True)
            self.y.copy_(hy, non_blocking=True)
        return self.run_round()

    @property
    def h2d_bytes_per_round(self) -> int:
        return self.host_x.numel() + self.host_y.numel() * 8

    @property
    def d2h_bytes_per_round(self) -> int:
        return self.out_host.numel() * 4
