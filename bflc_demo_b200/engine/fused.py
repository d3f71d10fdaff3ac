"""The B200-native round engine: one process per GPU, every rank replays the SAME captured
CUDA graph each round; who trains and who validates is decided by data in the HBM ledger
page (role bits), not by launch topology.

  round graph (all ranks; 7-8 launches):
    fed_plan_round  ||  prep_inputs    QueryState (local read of the ledger page); this round's
                                       inputs (u8 -> bf16, + e4m3 and scale chunks in fp8 mode) and
                                       the MXFP8 copy of the new global weights on a parallel branch
    [trainer]  mlp_round               the whole local epoch in ONE persistent kernel whose last
                                       optimizer epilogue IS UploadLocalUpdate (writes the upload
                                       buffers, releases FLAG_TRAINED on every peer)
                                       (csrc/kernels/mlp_round_sm100.cu; per-GEMM launches +
                                       fed_upload with ``fused_step=False``: models/mlp.py)
    [committee] fed_pull_*             QueryAllUpdates: each candidate's weights cross NVLink once
                                       (fp8: one 227 KB blob per candidate); BFLC_FUSED_PULL=1 moves
                                       this gather into the validation kernel itself
                mlp_val                validation of every candidate in one launch (or two grouped
                                       GEMMs whose TMA pulls the trainers' HBM directly)
    fed_consensus_aggregate            UploadScores + Aggregate + QueryGlobalModel

``cfg.dtype``: "bf16", or "fp8" = BASELINE.json config #2: fwd1/fwd2 of training and the whole
committee validation run block-scaled fp8 (tcgen05.mma.kind::mxf8f6f4.block_scale), gradients
bf16, master weights / Adam moments fp32.

No NCCL call and no host synchronisation inside a round.  The host C++ ledger drains the
device block ring afterwards and re-executes every election (``Ledger.AppendDeviceRound``).

Reference call stacks replaced: SURVEY.md 3.2 (trainer round) and 3.3 (committee round),
i.e. python-sdk/main.py:103-169, 196-228 and CommitteePrecompiled.cpp:215-456.
"""
from __future__ import annotations

import os

import struct
import time
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist

from .._native import C, ledger as _ledger
from ..config import FLConfig
from ..data.synthetic import Shard
from ..models.flat import ParamSpec
from ..models.mlp import FlatMLP, mlp_spec
from ..ops import gemm as G
from ..parallel.layout import HeapLayout
from ..parallel.symm import SymmetricHeap

ROLE_TRAINER, ROLE_COMM = 1, 2


def initial_roles(cfg: FLConfig) -> List[int]:
    """Genesis committee (reference: first COMM_COUNT entries in unordered_map order,
    C:176-182 -- arbitrary but deterministic): lowest ids, or a seeded permutation."""
    n = cfg.clients
    if cfg.solo:
        return [ROLE_TRAINER | ROLE_COMM] * n
    ids = list(range(n))
    if cfg.seed:
        rng = np.random.default_rng(cfg.seed)
        rng.shuffle(ids)
    roles = [ROLE_TRAINER] * n
    for i in ids[: cfg.committee_size]:
        roles[i] = ROLE_COMM
    return roles


# RoundState (csrc/include/bflc_kernels.h): epoch, n_ranks, n_comm, n_aggregate, role[8],
# last_median[8], selected_mask, global_loss, model_digest, blocks_appended, n_needed
_ROUND_STATE = struct.Struct("<4I8I8fIfQII")


class FusedEngine:
    def __init__(self, cfg: FLConfig, shard: Shard, *, rank: int = 0, world: int = 1,
                 device: int = 0, group=None, in_dim: Optional[int] = None):
        cfg.require_plain_fedavg("FusedEngine")
        assert cfg.clients == world, "one client per rank"
        assert world <= 8
        self.cfg, self.rank, self.world, self.device = cfg, rank, world, device
        self.group = group
        torch.cuda.set_device(device)
        self.dev = torch.device("cuda", device)
        self.mod = C()
        sz = self.mod.struct_sizes()
        self.sz = sz
        assert sz["RoundState"] == _ROUND_STATE.size, "RoundState layout changed: update _ROUND_STATE"

        # ---- model + heap --------------------------------------------------------------
        x0 = shard.x.reshape(len(shard), -1)
        self.in_dim = in_dim or x0.shape[1]
        self.spec: ParamSpec = mlp_spec(self.in_dim, cfg.hidden, shard.n_classes)
        self.n_params = self.spec.total
        self.S = (len(shard) // cfg.batch_size) * cfg.batch_size  # drop remainder (M:141)
        self.steps = (self.S // cfg.batch_size) * cfg.local_epochs
        self.n_val = min(cfg.val_samples or len(shard), len(shard))
        # block-scaled fp8: needs the persistent trainer's shape family (hidden 256, <= 64 classes)
        self.fp8 = cfg.dtype == "fp8"
        if self.fp8 and not (cfg.hidden == 256 and shard.n_classes <= 64 and cfg.fused_step
                             and cfg.batch_size % 128 == 0 and self.in_dim % 16 == 0
                             and len(shard) % 128 == 0):
            raise ValueError("dtype='fp8' (MXFP8) needs hidden == 256, <= 64 classes, batch % 128 == 0, "
                             "in_dim % 16 == 0, shard rows % 128 == 0 and the fused step")
        self.ql = self.mod.mx8_mlp_layout(self.in_dim, cfg.hidden) if self.fp8 else None
        self.blob_bytes = (self.ql["total"] + 4095) // 4096 * 4096 if self.fp8 else 0
        self.layout = HeapLayout(self.n_params, cfg.ring_slots, extra_bytes=2 * self.blob_bytes)
        self.heap = SymmetricHeap(self.layout.total_bytes, rank=rank, world=world, device=device,
                                  group=group, want_multicast=cfg.use_multicast)
        self.fed = self.layout.fed_dict(rank, world, self.heap.peer_ptrs, self.heap.mc_ptr)
        o = self.layout.offsets
        P = self.n_params
        hv = self.heap.view
        self.work_master = hv(o["work_master"], [P], torch.float32)
        self.work_shadow = hv(o["work_shadow"], [P], torch.bfloat16)
        self.global_master = hv(o["global"], [P], torch.float32)
        self.global_shadow = hv(o["global_shadow"], [P], torch.bfloat16)
        self.state_bytes = hv(o["state"], [sz["RoundState"]], torch.uint8)
        self.plan_bytes = hv(o["plan"], [sz["RoundPlan"]], torch.uint8)
        self.ring_bytes = hv(o["ring"], [cfg.ring_slots * sz["BlockRecord"]], torch.uint8)
        plan_ptr = self.heap.local_ptr + o["plan"]
        self.plan_ptr = plan_ptr
        self.is_trainer_ptr = plan_ptr + sz["plan_is_trainer_off"]
        self.is_comm_ptr = plan_ptr + sz["plan_is_comm_off"]
        self.loss_sum = hv(o["plan"] + sz["plan_loss_sum_off"], [1], torch.float32)
        self.train_correct = hv(o["plan"] + sz["plan_train_correct_off"], [1], torch.int32)
        self.val_correct = hv(o["plan"] + sz["plan_correct_off"], [sz["kMaxRanks"]], torch.int32)
        self.grad = torch.zeros(P, device=self.dev, dtype=torch.float32)

        # genesis model: identical on every rank
        init = torch.empty(P, dtype=torch.float32)
        self.spec.init_(init, seed=cfg.seed + 1234)
        for t in (self.work_master, self.global_master):
            t.copy_(init)
        for t in (self.work_shadow, self.global_shadow):
            t.copy_(init.to(torch.bfloat16))

        # ledger page + host chain
        roles = initial_roles(cfg)
        st = self.mod.state_init_bytes(world, cfg.committee_size, cfg.aggregate_count, roles,
                                       cfg.needed_updates)
        self.state_bytes.copy_(torch.frombuffer(bytearray(st), dtype=torch.uint8))
        self.host_ledger = _ledger().Ledger(cfg.to_ledger_config(P))
        self.host_ledger.Bootstrap(roles)
        self.drained = 0

        # ---- model trainer over heap views -----------------------------------------------
        self.trainer = FlatMLP(self.spec, self.work_master, self.work_shadow, self.grad,
                               cfg.batch_size, optimizer=cfg.optimizer, lr=cfg.learning_rate,
                               loss_sum=self.loss_sum, correct=self.train_correct,
                               step_dev_ptr=plan_ptr + sz["plan_opt_step_off"], fp8=self.fp8)
        # upload buffers start as the genesis model (the fused upload never touches the padding
        # elements between tensors; FedAvg must not sum garbage there)
        for par in (0, 1):
            hv(o[f"upload_master{par}"], [P], torch.float32).copy_(init)
            hv(o[f"upload_shadow{par}"], [P], torch.bfloat16).copy_(init.to(torch.bfloat16))
        self.upq_off = [o["extra"], o["extra"] + self.blob_bytes] if self.fp8 else []
        if self.fp8:
            for off in self.upq_off:
                self.trainer.quantize_weights(self.global_master, hv(off, [self.blob_bytes], torch.uint8))
            self.trainer.quantize_weights()

        # ---- data ------------------------------------------------------------------------
        self.x_u8 = torch.empty(len(shard), self.in_dim, device=self.dev, dtype=torch.uint8)
        self.x_bf = torch.empty(len(shard), self.in_dim, device=self.dev, dtype=torch.bfloat16)
        if self.fp8:
            from ..models.mlp import sf_bytes
            self.x_q = torch.zeros(len(shard), self.in_dim, device=self.dev, dtype=torch.uint8)
            self.x_sf = torch.full((sf_bytes(len(shard), self.in_dim),), 127, device=self.dev,
                                   dtype=torch.uint8)
        else:
            self.x_q = self.x_sf = None
        self.y = torch.empty(len(shard), device=self.dev, dtype=torch.int32)
        self.host_x = x0.contiguous().pin_memory()
        self.host_y = shard.y.to(torch.int32).contiguous().pin_memory()
        self.x_u8.copy_(self.host_x)
        self.y.copy_(self.host_y)
        self.h_val = torch.empty(world, self.n_val, cfg.hidden, device=self.dev, dtype=torch.bfloat16)
        self.out_host = torch.empty(sz["RoundState"], dtype=torch.uint8).pin_memory()
        self.rec_host = torch.empty(sz["BlockRecord"], dtype=torch.uint8).pin_memory()

        # ---- validation tensor-map table [layer][parity][rank] (peers' upload shadows) ----
        K = sz["kMaxRanks"]
        e1, e2 = self.spec.by_name["w1"], self.spec.by_name["w2"]
        # N-tile widths are pinned so the pre-encoded peer tensor maps match the launches
        self.val_bn = [self.mod.gemm_pick_bn(e1.shape[0], G.EPI_GENERIC, self.n_val, world),
                       self.mod.gemm_pick_bn(e2.shape[0], G.EPI_ARGMAX, self.n_val, world)]
        # hidden == 256: the whole validation forward of every candidate is ONE launch
        # (mlp_val_sm100: fwd1 -> relu -> fwd2 -> argmax per (128 rows, candidate) CTA, hidden
        # activations stay in TMEM / smem); its layer-1 maps use a 256-row box.
        self.val_chain = (cfg.hidden == 256 and e2.shape[0] <= 64
                          and os.environ.get("BFLC_VAL_CHAIN", "1") != "0")
        if self.val_chain:
            self.val_bn = [256, 64]
        # Two ways to feed the candidates' weights to the validation GEMMs:
        #  staged (default): fed_pull_candidates streams each trainer's bf16 weights out of its
        #    HBM once (as soon as that trainer's flag is up); the GEMM B maps cover the local
        #    staging slots [layer][slot].
        #  direct: the B maps cover the trainers' upload buffers [layer][parity][rank] and the
        #    GEMM's TMA producer pulls tiles across NVLink itself -- no staging pass, but every
        #    M-tile CTA re-reads the weights remotely (good only for few M-tiles).
        self.staged = bool(cfg.stage_candidates) and world > 1
        if self.fp8:
            self.cand_q = torch.zeros(world, self.blob_bytes, device=self.dev, dtype=torch.uint8)
            self.cand_shadow = None
        else:
            self.cand_q = None
            self.cand_shadow = torch.zeros(world, P, device=self.dev, dtype=torch.bfloat16)
        blob = bytearray(2 * 2 * K * 128)

        def b_map(base, e, kind, layer):
            if self.fp8:   # e4m3 rows inside an Mx8MlpLayout blob; W2 is padded to 64 rows
                rows = e.shape[0] if layer == 0 else 64
                return self.mod.gemm_b_map(base + self.ql["w1q" if layer == 0 else "w2q"], rows,
                                           e.shape[1], e.shape[1], False, True, kind, self.val_bn[layer])
            return self.mod.gemm_b_map(base + e.offset * 2, e.shape[0], e.shape[1], e.shape[1], False,
                                       False, kind, self.val_bn[layer])

        for layer, (e, kind) in enumerate(((e1, G.EPI_GENERIC), (e2, G.EPI_ARGMAX))):
            if self.staged:
                for zslot in range(world):
                    base = (self.cand_q.data_ptr() + zslot * self.blob_bytes if self.fp8
                            else self.cand_shadow.data_ptr() + zslot * P * 2)
                    idx = layer * K + zslot
                    blob[idx * 128:(idx + 1) * 128] = b_map(base, e, kind, layer)
                continue
            for par in range(2):
                for r in range(world):
                    base = self.heap.peer_ptrs[r] + (self.upq_off[par] if self.fp8
                                                     else o[f"upload_shadow{par}"])
                    idx = (layer * 2 + par) * K + r
                    blob[idx * 128:(idx + 1) * 128] = b_map(base, e, kind, layer)
        self.b_maps = torch.frombuffer(blob, dtype=torch.uint8).to(self.dev)
        self.plan_layers = [(self.spec.offset("b1"), True), (self.spec.offset("b2"), True)]
        self.dyn_ptr = [plan_ptr + sz["plan_dyn_off"] + i * sz["GemmDynamic"] for i in range(2)]
        # FedAvg as "every rank reduces everything" (one-shot) or "reduce my 1/n slice, publish it
        # to all replicas" (two-shot).  Measured on the 0.87 MB model: two-shot 3301 vs 2988
        # rounds/s at 8 GPUs (8 ranks each pulling 4 whole uploads contend with the committee's
        # pulls), 3612 vs 3671 at 4 GPUs -> two-shot from 8 ranks up, and always for big models.
        self.two_shot = (cfg.two_shot if cfg.two_shot is not None
                         else world > 1 and (P * 4 > (64 << 20) or world >= 8))
        self.byz = 1 if rank in cfg.byzantine_ranks else 0
        self.straggle_us = cfg.straggler_delay_us if rank in cfg.straggler_ranks else 0
        # first-K-wins admission (needed_updates < trainers): candidate slots are resolved on the
        # device from the admission tickets, which needs the staged (pull) validation path
        self.first_k = (not cfg.solo) and cfg.needed_updates < cfg.n_trainers
        if self.first_k and not self.staged:
            raise ValueError("needed_updates < trainers (first-K-wins admission) needs stage_candidates=True")
        # Hot path 1 as ONE kernel (opt-in, BFLC_FUSED_PULL=1): the validation CTAs gather the
        # candidates' MXFP8 blobs out of the trainers' HBM themselves (mlp_val_sm100.cu).  Correct
        # (multi_gpu_check fused / fedavg / byzantine) but measured 4 us per round SLOWER than the
        # separate pull kernel at 2 GPUs (249.7 vs 244.3 us, profiles/r2/bench_n2_fused_pull_ab_*.log):
        # k_pull_blob is already resident and spinning on the trainers' flags when they arrive and
        # its tail overlaps the validation kernel's prologue (PDL), while the in-kernel gather adds
        # a P2P round trip plus a counter barrier to every validation CTA.  Default: separate pull.
        # first-K mode always keeps the pull kernel (slot -> trainer is only known from the tickets).
        self.fused_pull = (self.fp8 and self.staged and not self.first_k and (self.n_val + 127) // 128 <= 128
                           and os.environ.get("BFLC_FUSED_PULL", "0") == "1")
        self.fused_step = bool(cfg.fused_step) and self.trainer.fused_ok(self.steps)
        # UploadLocalUpdate inside the trainer's last optimizer epilogue (needs E_OPT)
        self.fused_upload = self.fused_step and os.environ.get("BFLC_MLP_EPIOPT", "1") != "0"
        if self.fp8 and not (self.fused_step and self.fused_upload):
            raise ValueError("dtype='fp8' needs the persistent trainer with the optimizer epilogue")
        self._rounds = 0
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.graph_pipe: Optional[torch.cuda.CUDAGraph] = None
        self._exec: Dict[int, int] = {}
        self.stream = torch.cuda.Stream(device=self.dev)
        self._side = torch.cuda.Stream(device=self.dev)
        self._side2 = torch.cuda.Stream(device=self.dev)
        self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
        # host -> device input pipeline (run_round_e2e): needs the one-launch trainer (its producer
        # waits per step) and a shard that is exactly steps x batch rows
        self.pipelined_input = (self.fused_step and self.S == len(shard) and self.steps <= 16
                                and (cfg.batch_size * self.in_dim) % 16 == 0
                                and os.environ.get("BFLC_INPUT_PIPELINE", "1") != "0"
                                and os.environ.get("BFLC_MLP_CHAIN", "3") != "1")
        # result read-back of run_round_e2e: the consensus kernel mirrors the committed ledger page
        # into this pinned page and release-stores the new epoch into word MIRROR_SEQ; the host
        # polls it (no copy-engine launch, no stream sync at the end of a round)
        self.mirror = torch.zeros(128, dtype=torch.int32).pin_memory()
        self._mirror_np = self.mirror.numpy()
        self._epoch_known: Optional[int] = None
        self.mirror_result = os.environ.get("BFLC_RESULT_MIRROR", "1") != "0"
        self.in_flags = torch.zeros(16, device=self.dev, dtype=torch.int32)
        self.in_seq = torch.zeros(1, device=self.dev, dtype=torch.int32)
        self.cast_cnt = torch.zeros(16, device=self.dev, dtype=torch.int32)
        self.x_ready = torch.zeros(16, device=self.dev, dtype=torch.int32)
        self.in_err = torch.zeros(1, device=self.dev, dtype=torch.int32)
        self._ev_wq = torch.cuda.Event()
        self.seq_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self._seq_np = self.seq_host.numpy()
        self._seq = 0
        self._copy_stream = torch.cuda.Stream(device=self.dev)
        # constant arguments of the per-round h2d_pipeline call (kept off the per-round Python path)
        self._pipe_dst, self._pipe_y = self.x_u8.data_ptr(), self.y.data_ptr()
        self._pipe_chunk = self.cfg.batch_size * self.in_dim
        self._pipe_flags = (self.in_flags.data_ptr(), self.seq_host.data_ptr(), self._copy_stream.cuda_stream)
        self._prefeed = os.environ.get("BFLC_E2E_PREFEED", "1") == "1"
        self._tag_wv = os.environ.get("BFLC_E2E_TAGS", "writevalue") != "memcpy"
        self.launches_per_round = 0
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize()

    # ------------------------------------------------------------------ one round
    def _enqueue_round(self, pipe: bool = False):
        """One round.  ``pipe``: the input-pipeline variant used by ``run_round_e2e`` (chunked,
        tag-driven input conversion overlapping the training steps); the plain variant converts
        the resident inputs up front.  Both leave identical state."""
        m, cfg = self.mod, self.cfg
        pipe = pipe and self.pipelined_input
        n0 = m.launch_count()
        # The input cast does not depend on the plan: it runs as a parallel branch of the captured
        # graph.  With the input pipeline it is a persistent kernel that converts chunk s (the rows
        # of local step s) as soon as that chunk's H2D copy has landed (run_round_e2e), and the
        # trainer's TMA producer waits per step -- the branch is joined only before validation.
        main = torch.cuda.current_stream()
        self._ev_fork.record(main)
        self._side.wait_event(self._ev_fork)
        B = cfg.batch_size
        if self.fp8:
            # the consensus kernel of the previous round rewrote the training weights: refresh this
            # trainer's MXFP8 copy (e4m3 + scale chunks) before step 0 -- a third parallel branch
            self._side2.wait_event(self._ev_fork)
            with torch.cuda.stream(self._side2):
                self.trainer.quantize_weights()
                self._ev_wq.record(self._side2)
        with torch.cuda.stream(self._side):
            if pipe:
                m.prep_inputs_chunks(self.x_u8, self.x_bf, self.x_q, self.x_sf, B, self.steps,
                                     1.0 / 255.0, self.in_flags, self.in_seq, self.cast_cnt,
                                     self.x_ready, self.in_err)
            else:
                m.prep_inputs(self.x_u8, self.x_bf, self.x_q, self.x_sf, 1.0 / 255.0)
            self._ev_join.record(self._side)
        if self.fp8:
            m.fed_plan_round(self.fed, self.plan_layers, self.steps, self.staged,
                             self.cand_q.data_ptr(), self.blob_bytes, self.upq_off, self.fused_pull)
        else:
            m.fed_plan_round(self.fed, self.plan_layers, self.steps, self.staged)
        if not pipe:
            main.wait_event(self._ev_join)
        if self.fp8:
            main.wait_event(self._ev_wq)
        # local training, predicated on the trainer role bit
        m.set_predicate(self.is_trainer_ptr)
        if self.fused_step:
            # every local step of the round inside ONE persistent kernel (phase barriers instead
            # of launches); the barrier word lives in the plan and is zeroed by k_plan.  With
            # fused_upload its last optimizer epilogue publishes the update (UploadLocalUpdate).
            up = dict(fed=self.fed, upq_off=self.upq_off, n_samples=self.S,
                      n_loss_terms=self.steps * B, byz_mode=self.byz,
                      byz_scale=cfg.byzantine_scale, straggle_us=self.straggle_us) if self.fused_upload else {}
            self.trainer.train_epoch_fused(
                self.x_bf, self.y, self.steps, self.plan_ptr + self.sz["plan_step_barrier_off"],
                None, -1, -1,
                self.x_ready.data_ptr() if pipe else 0, self.in_seq.data_ptr() if pipe else 0,
                x_q=self.x_q, x_sf=self.x_sf, **up)
        else:
            self.trainer.train_epoch(self.x_bf, self.y, self.steps)
        m.set_predicate(0)
        if pipe:
            main.wait_event(self._ev_join)      # validation reads every converted row
        if not (self.fused_step and self.fused_upload):
            m.fed_upload(self.fed, self.S, self.steps * B, self.byz, cfg.byzantine_scale, self.straggle_us)
        # committee validation: grouped GEMMs whose B operands are the trainers' uploads
        if self.staged:
            if self.fused_pull:
                pass        # QueryAllUpdates happens inside the validation kernel (fused gather)
            elif self.fp8:
                m.fed_pull_blobs(self.fed, self.upq_off[0], self.upq_off[1], self.blob_bytes, self.cand_q)
            else:
                m.fed_pull_candidates(self.fed, self.cand_shadow, None)
        H = cfg.hidden
        if self.fp8:
            m.set_predicate(self.is_comm_ptr)
            m.mlp_val(self.x_q[: self.n_val], self.y[: self.n_val], self.val_correct, self.b_maps,
                      self.dyn_ptr[0], self.dyn_ptr[1], self.n_val, self.in_dim, H,
                      self.spec.by_name["w2"].shape[0], self.world, self.x_sf,
                      self.plan_ptr + self.sz["plan_cand_blob_off"],
                      *((self.plan_ptr + self.sz["plan_cand_src_off"], self.plan_ptr + self.sz["plan_pull_cnt_off"],
                         self.blob_bytes, self.plan_ptr + self.sz["plan_stamps_off"]) if self.fused_pull else ()))
            m.set_predicate(0)
        else:
            xv, yv = self.x_bf[: self.n_val], self.y[: self.n_val]
            if self.val_chain:
                m.set_predicate(self.is_comm_ptr)
                m.mlp_val(xv, yv, self.val_correct, self.b_maps, self.dyn_ptr[0], self.dyn_ptr[1],
                          self.n_val, self.in_dim, H, self.spec.by_name["w2"].shape[0], self.world)
                m.set_predicate(0)
            else:
                self._validate_two_gemms(xv, yv, H)
        m.fed_consensus_aggregate(self.fed, self.n_val, cfg.weight_by_score, self.two_shot,
                                  cfg.use_multicast and self.heap.has_multicast,
                                  self.mirror.data_ptr() if (pipe and self.mirror_result) else 0,
                                  self.in_seq.data_ptr() if pipe else 0)
        self.launches_per_round = int(m.launch_count() - n0)

    def _validate_two_gemms(self, xv, yv, H):
        m = self.mod
        m.gemm(xv, self.work_shadow, self.h_val, self.n_val, H, self.in_dim, self.world,
               self.in_dim, self.in_dim, 0, 0, False, False, False, G.EPI_GENERIC, 1, H,
               self.n_val * H, 1.0, None, G.ACT_RELU, None, None, 0, None, 1, False, None, 0, 1.0,
               None, None, self.b_maps, None, 0, 0, 0, 0, self.dyn_ptr[0], self.val_bn[0])
        m.gemm(self.h_val, self.work_shadow, None, self.n_val, self.spec.by_name["w2"].shape[0], H,
               self.world, H, H, self.n_val * H, 0, False, False, False, G.EPI_ARGMAX, 1, 0, 0, 1.0,
               None, 0, None, None, 0, None, 1, False, yv, 0, 1.0, None, self.val_correct,
               self.b_maps, None, 0, 0, 0, 0, self.dyn_ptr[1], self.val_bn[1])

    def capture(self):
        """Warm up eagerly (lazy kernel attribute setup), then capture one round."""
        with torch.cuda.stream(self.stream):
            self._enqueue_round()
        self.stream.synchronize()
        self._rounds += 1          # the warm-up is a real round (epoch advanced)
        if not self.cfg.cuda_graph:
            return
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self.stream):
            self._enqueue_round()
        self.graph = g
        if self.pipelined_input:
            # second graph for run_round_e2e: same round, inputs converted chunk by chunk as
            # their H2D copies land.  Its only new kernel is warmed up once outside the capture
            # (lazy module loading), without running an extra round.
            with torch.cuda.stream(self.stream):
                self.in_seq.fill_(-1)       # the kernel waits for tag *in_seq + 1: 0 = the initial tags
                self.mod.prep_inputs_chunks(self.x_u8, self.x_bf, self.x_q, self.x_sf,
                                            self.cfg.batch_size, self.steps, 1.0 / 255.0,
                                            self.in_flags, self.in_seq, self.cast_cnt, self.x_ready,
                                            self.in_err)
                self.in_seq.zero_()         # rounds fed so far (bumped by the consensus kernel)
            self.stream.synchronize()
            gp = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gp, stream=self.stream):
                self._enqueue_round(pipe=True)
            self.graph_pipe = gp
        # raw executable handles for the per-round launch (the captured rounds use no torch RNG, so
        # CUDAGraph.replay()'s generator prologue has nothing to do)
        self._stream_ptr = self.stream.cuda_stream
        if os.environ.get("BFLC_RAW_GRAPH_LAUNCH", "1") != "0":
            for gg in (self.graph, self.graph_pipe):
                try:
                    if gg is not None:
                        self._exec[id(gg)] = int(gg.raw_cuda_graph_exec())
                except Exception:      # older torch: fall back to replay()
                    pass

    def run_round(self, pipe: bool = False):
        # the device BlockRecord ring has ring_slots entries and the consensus kernel overwrites
        # slot epoch % ring_slots: drain into the host ledger before records can be lost
        self._rounds += 1
        if self._epoch_known is not None:
            self._epoch_known += 1          # every round advances the epoch by exactly one
        if self._rounds - self.drained >= max(self.cfg.ring_slots // 2, 1):
            errs = self.drain_blocks()
            if errs:
                raise RuntimeError(f"host/device ledgers disagree: {errs[:2]}")
        g = self.graph_pipe if (pipe and self.graph_pipe is not None) else self.graph
        if g is not None:
            ex = self._exec.get(id(g))
            if ex:      # cudaGraphLaunch straight on the engine stream (no guard, no replay bookkeeping)
                self.mod.graph_launch(ex, self._stream_ptr)
            else:
                with torch.cuda.stream(self.stream):
                    g.replay()
        else:
            with torch.cuda.stream(self.stream):
                self._enqueue_round(pipe=pipe)

    def run_round_e2e(self, host_x: Optional[torch.Tensor] = None,
                      host_y: Optional[torch.Tensor] = None) -> dict:
        """Public per-round call: stage this round's inputs from pinned host memory, run the
        round, read the result (ledger page) back to the host."""
        hx = self.host_x if host_x is None else host_x
        hy = self.host_y if host_y is None else host_y
        if self.pipelined_input:
            # launch the round first, then feed it: labels, chunk 0, tag 0, chunk 1, tag 1, ... on
            # the copy stream; step s of the trainer starts when chunk s has been converted, so
            # the copy of the later chunks hides behind the compute of the earlier steps
            # The copies of round r carry tag r; the device counts fed rounds itself (the consensus
            # kernel bumps in_seq at the end of every pipelined round), so nothing has to be
            # copied in front of the graph.
            self._seq += 1
            self._seq_np[0] = self._seq
            # launch the round, then feed it (measured: issuing chunk 0 ahead of the graph launch
            # was slower, profiles/run27_*)
            yb = hy.numel() * hy.element_size()
            if self._prefeed:   # labels + chunk 0 travel while the graph launch is in progress
                self.mod.h2d_pipeline(hx.data_ptr(), self._pipe_dst, self._pipe_chunk, 0, 1,
                                      hy.data_ptr(), self._pipe_y, yb, *self._pipe_flags, self._tag_wv)
                self.run_round(pipe=True)
                self.mod.h2d_pipeline(hx.data_ptr(), self._pipe_dst, self._pipe_chunk, 1, self.steps,
                                      0, 0, 0, *self._pipe_flags, self._tag_wv)
            else:
                self.run_round(pipe=True)
                self.mod.h2d_pipeline(hx.data_ptr(), self._pipe_dst, self._pipe_chunk, 0, self.steps,
                                      hy.data_ptr(), self._pipe_y, yb, *self._pipe_flags, self._tag_wv)
        else:
            with torch.cuda.stream(self.stream):
                self.x_u8.copy_(hx, non_blocking=True)
                self.y.copy_(hy, non_blocking=True)
            self.run_round()
        if self.pipelined_input and self.mirror_result and self.graph_pipe is not None \
                and self._epoch_known is not None:
            # the kernel wrote the page into pinned memory; every chunk copy was consumed before
            # the trainer's last step, so nothing is in flight once the new epoch is visible
            self._wait_mirror(self._epoch_known)
            return self.read_state(self.mirror)
        with torch.cuda.stream(self.stream):
            self.out_host.copy_(self.state_bytes, non_blocking=True)
        self.stream.synchronize()
        if self.pipelined_input:
            self._copy_stream.synchronize()
        st = self.read_state(self.out_host)
        self._epoch_known = st["epoch"]
        return st

    def _wait_mirror(self, want: int):
        m, n, t0 = self._mirror_np, 0, None
        seq = int(self.sz["kMirrorSeqWord"])
        while int(m[seq]) != want:
            n += 1
            if (n & 0x3FFF) == 0:
                now = time.monotonic()
                if t0 is None:
                    t0 = now
                elif now - t0 > 30.0:
                    raise RuntimeError(f"round result never reached the host mirror page (want epoch {want}, "
                                       f"have {int(m[seq])})")

    @property
    def h2d_bytes_per_round(self) -> int:
        tags = 4 * self.steps if self.pipelined_input else 0   # one 4-byte tag per chunk
        return self.host_x.numel() * self.host_x.element_size() + self.host_y.numel() * 4 + tags

    @property
    def d2h_bytes_per_round(self) -> int:
        if self.pipelined_input and self.mirror_result:
            return int(self.sz["RoundState"]) + 4      # ledger page + epoch word, written by the kernel
        return self.out_host.numel()

    # ------------------------------------------------------------------ host views
    def read_state(self, buf: Optional[torch.Tensor] = None) -> dict:
        if buf is not None and buf is getattr(self, "mirror", None):   # (GenericFedEngine borrows this method)
            # hot path of run_round_e2e: one precompiled unpack straight out of the pinned page
            f = _ROUND_STATE.unpack_from(self._mirror_np, 0)
            w = self.world
            return dict(epoch=f[0], roles=list(f[4:4 + w]), median=list(f[12:12 + w]), selected_mask=f[20],
                        global_loss=f[21], model_digest=f[22])
        else:
            b = bytes((self.state_bytes.cpu() if buf is None else buf).numpy())
        epoch, n_ranks, n_comm, n_agg = struct.unpack_from("<4I", b, 0)
        roles = list(struct.unpack_from("<8I", b, 16))[: self.world]
        med = list(struct.unpack_from("<8f", b, 48))[: self.world]
        sel, = struct.unpack_from("<I", b, 80)
        loss, = struct.unpack_from("<f", b, self.sz["state_global_loss_off"])
        digest, = struct.unpack_from("<Q", b, self.sz["state_digest_off"])
        return dict(epoch=epoch, roles=roles, median=med, selected_mask=sel, global_loss=loss,
                    model_digest=digest)

    def read_stamps(self) -> dict:
        """%globaltimer phase stamps (ns) of the LAST finished round on this rank, turned into
        durations (us).  ``exposed_comm_us`` = upload + candidate pull + consensus/FedAvg/publish,
        i.e. everything in the round that is neither local training nor the validation GEMMs."""
        torch.cuda.synchronize()
        raw = bytes(self.plan_bytes.cpu().numpy())
        t = struct.unpack_from("<8Q", raw, self.sz["plan_stamps_off"])

        def d(a, b):
            return (t[b] - t[a]) / 1e3 if t[a] and t[b] and t[b] >= t[a] else 0.0
        out = dict(train_us=d(0, 1) if t[1] else 0.0, upload_us=d(1, 2), pull_us=d(3, 4),
                   # direct (unstaged) validation has no pull stamps: it starts after the upload
                   validate_us=d(4, 5) if t[4] else (d(2, 5) if t[2] else 0.0),
                   consensus_wait_us=d(5, 6),
                   aggregate_publish_us=d(6, 7), round_us=d(0, 7))
        # pull_us on a committee rank includes waiting for the trainers' flags (it starts with
        # the round); the exposed part is what is left of the round after compute
        out["exposed_comm_us"] = max(out["round_us"] - out["train_us"] - out["validate_us"], 0.0)
        return out

    def drain_blocks(self) -> List[str]:
        """Pull finished BlockRecords off the device ring into the host C++ ledger, which
        re-executes each election.  Returns the list of mismatches ([] = replicas agree)."""
        torch.cuda.synchronize()
        if getattr(self, "in_err", None) is not None and int(self.in_err.item()):
            raise RuntimeError("input pipeline: a chunk's H2D tag never arrived (host stalled > 10 s "
                               "between launching the round and feeding it); the round ran on stale inputs")
        st = self.read_state()
        ring = bytes(self.ring_bytes.cpu().numpy())
        rs = self.sz["BlockRecord"]
        errs = []
        K = 8
        while self.drained < st["epoch"]:
            e = self.drained
            off = (e % self.cfg.ring_slots) * rs
            rec = ring[off:off + rs]
            f = struct.unpack_from("<4I", rec, 0)
            p = 16
            role_before = list(struct.unpack_from("<8I", rec, p)); p += 32
            role_after = list(struct.unpack_from("<8I", rec, p)); p += 32
            rows = [list(struct.unpack_from("<8f", rec, p + 32 * c)) for c in range(K)]; p += 256
            scored = list(struct.unpack_from("<8I", rec, p)); p += 32
            p += 32  # median
            n_samples = list(struct.unpack_from("<8I", rec, p)); p += 32
            avg_cost = list(struct.unpack_from("<8f", rec, p)); p += 32
            p += 32  # weight
            adm, sel = struct.unpack_from("<2I", rec, p); p += 8
            gl, = struct.unpack_from("<f", rec, p); p += 4
            wbs, = struct.unpack_from("<I", rec, p); p += 4
            digest, = struct.unpack_from("<Q", rec, p); p += 8
            seq, = struct.unpack_from("<I", rec, p)
            if f[0] != e or seq != e + 1:
                errs.append(f"ring slot for epoch {e} holds epoch {f[0]} seq {seq}")
                break
            n = self.world
            msg = self.host_ledger.AppendDeviceRound(dict(
                epoch=e, role_before=role_before[:n], role_after=role_after[:n],
                score_rows=[r[:n] for r in rows[:n]], scored_mask=scored[:n],
                n_samples=n_samples[:n], avg_cost=avg_cost[:n], admitted_mask=adm,
                selected_mask=sel, global_loss=gl, model_digest=digest, weight_by_score=wbs))
            if msg:
                errs.append(f"epoch {e}: {msg}")
                break
            self.drained += 1
        return errs

    def global_model(self) -> Dict[str, torch.Tensor]:
        return {k: v.clone() for k, v in self.spec.views(self.global_master).items()}

    def evaluate(self, shard: Shard) -> float:
        """Sponsor-style test accuracy of the current global model (M:285-306)."""
        x = shard.x.reshape(len(shard), -1).to(self.dev)
        xb = torch.empty(x.shape, device=self.dev, dtype=torch.bfloat16)
        self.mod.prep_inputs(x.contiguous(), xb, None, None, 1.0 / 255.0)
        cnt = self.trainer.accuracy_counts(xb, shard.y.to(self.dev, torch.int32),
                                           shadow=self.global_shadow, master=self.global_master)
        return float(cnt.item()) / len(shard)
