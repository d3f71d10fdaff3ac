"""Command-line runner for the GPU engines (the counterpart of ``python main.py`` in the
reference, python-sdk/main.py:343-358, for one NVSwitch box):

    python -m bflc_demo_b200.run --model mlp --rounds 20                       # 1 GPU, solo
    python -m bflc_demo_b200.run --clients 20 --rounds 20     # 20 clients on 1 GPU (20/4/10/6)
    python -m bflc_demo_b200.run --clients 20 --alpha 0.5 --size-sigma 0.8    # skewed labels + sizes
    python -m bflc_demo_b200.run --clients 20 --alpha 0.1 --prox-mu 0.01 --server-opt adam \
        --server-lr 0.01                                  # FedProx clients + FedAdam server
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 \\
        -m bflc_demo_b200.run --model resnet18 --rounds 5 --byzantine 7       # config #4

BASELINE.json configs: ``--model mlp`` (#2), ``lenet5`` (#3, non-IID CIFAR shards), ``resnet18``
(#4, use --byzantine), ``bert`` (#5, seq_len 128).  Rank 0 doubles as the sponsor: after every
round it evaluates the global model on a held-out test shard and prints the reference's two
log lines (``the E epoch , global loss : L`` / ``Epoch: 00E, test_acc: A``).
"""
from __future__ import annotations

import argparse
import json
import os
import time

import torch
import torch.distributed as dist

from .config import FLConfig
from .data.synthetic import cifar_like, client_sizes, femnist_like, tokens_like
from .utils.metrics import RunLog
from .utils.tracing import PhaseTimer


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="mlp", choices=["mlp", "lenet5", "resnet18", "bert"])
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--samples", type=int, default=0, help="samples per client (0 = model default)")
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--lr", type=float, default=0.0)
    ap.add_argument("--optimizer", default="sgd", choices=["sgd", "adam"])
    ap.add_argument("--byzantine", type=int, nargs="*", default=[])
    ap.add_argument("--bert-layers", type=int, default=12)
    ap.add_argument("--checkpoint", default="")
    ap.add_argument("--resume", default="")
    ap.add_argument("--no-stage", action="store_true", help="validate straight out of peers' HBM")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp8"],
                    help="fp8: block-scaled (MXFP8) forward GEMMs (the MLP keeps the fused persistent trainer)")
    ap.add_argument("--generic", action="store_true", help="run the MLP through GenericFedEngine")
    ap.add_argument("--clients", type=int, default=0,
                    help="clients (default: one per GPU); more than WORLD_SIZE on one GPU runs the "
                         "MLP through MultiClientEngine")
    ap.add_argument("--committee", type=int, default=4, help="--clients: committee size (COMM_COUNT)")
    ap.add_argument("--needed", type=int, default=10, help="--clients: NEEDED_UPDATE_COUNT")
    ap.add_argument("--aggregate", type=int, default=6, help="--clients: AGGREGATE_COUNT")
    ap.add_argument("--alpha", type=float, default=0.0,
                    help="--clients: Dirichlet label skew of every client (0 = IID)")
    ap.add_argument("--size-sigma", type=float, default=0.0,
                    help="--clients: log-normal spread of the shard sizes (0 = equal shards; the "
                         "total stays clients x samples)")
    fo = ap.add_argument_group("FedProx and server optimizers (--clients only)")
    fo.add_argument("--prox-mu", type=float, default=None,
                    help="FedProx: add mu/2 ||w - w_global||^2 to every client's local loss (default 0)")
    fo.add_argument("--server-opt", default=None, choices=["none", "momentum", "adam", "yogi"],
                    help="server step on the pseudo-gradient average - global (default none = FedAvg)")
    fo.add_argument("--server-lr", type=float, default=None, help="server learning rate (default 1.0)")
    fo.add_argument("--server-beta1", type=float, default=None, help="default 0.9")
    fo.add_argument("--server-beta2", type=float, default=None, help="default 0.99")
    fo.add_argument("--server-tau", type=float, default=None, help="adaptivity (default 1e-3)")
    a = ap.parse_args(argv)
    fedopt = {k: v for k, v in (("prox_mu", a.prox_mu), ("server_optimizer", a.server_opt),
                                 ("server_lr", a.server_lr), ("server_beta1", a.server_beta1),
                                 ("server_beta2", a.server_beta2), ("server_tau", a.server_tau))
              if v is not None}
    if fedopt and a.clients < 2:
        ap.error("--prox-mu and --server-* need --clients N (N >= 2): only the multi-client engine "
                 "implements FedProx and the server optimizers")
    a.fedopt = fedopt

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    lr_ = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(lr_)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr_))

    if a.clients > world:
        if world > 1:
            raise SystemExit(f"--clients {a.clients} > WORLD_SIZE {world}: several clients per GPU is "
                             "supported on a single GPU only")
        return run_multiclient(a)

    defaults = dict(mlp=(4096, 512, 0.05), lenet5=(2048, 128, 0.05), resnet18=(512, 64, 0.02),
                    bert=(64, 16, 0.002))[a.model]
    S, B, LR = a.samples or defaults[0], a.batch or defaults[1], a.lr or defaults[2]
    cfg = FLConfig.for_world(world, model=a.model, batch_size=B, samples_per_client=S,
                             learning_rate=LR, optimizer=a.optimizer, byzantine_ranks=a.byzantine,
                             stage_candidates=not a.no_stage, ring_slots=1024, dtype=a.dtype)
    if a.model == "mlp":
        shard = femnist_like(world, S, seed=7, only=rank)[0]
        test = femnist_like(1, 2048, seed=7, only=0)[0]
    elif a.model in ("lenet5", "resnet18"):
        shard = cifar_like(world, S, seed=7, alpha=0.5)[rank]
        test = cifar_like(1, 1024, seed=7, alpha=0.0)[0]
    else:
        shard = tokens_like(world, S, seed=7)[rank]
        test = tokens_like(1, 128, seed=8)[0]

    if a.model == "mlp" and not a.generic:
        from .engine.fused import FusedEngine
        eng = FusedEngine(cfg, shard, rank=rank, world=world, device=lr_)
        eng.capture()
    else:
        from .engine.generic import GenericFedEngine
        from .models.nets import build_model
        net = build_model(a.model, shard.n_classes, layers=a.bert_layers)
        eng = GenericFedEngine(cfg, net, shard, rank=rank, world=world, device=lr_)
    if a.resume:
        from .utils.checkpoint import load_checkpoint
        print(f"[rank {rank}] resumed:", load_checkpoint(a.resume, eng))

    log = RunLog(rank=rank)
    timer = PhaseTimer()
    t0 = time.time()
    for _ in range(a.rounds):
        with timer.phase("round"):
            eng.run_round()
        st = eng.read_state()
        acc = eng.evaluate(test) if rank == 0 else None        # sponsor (M:280-340)
        log.round(st["epoch"] - 1, st["global_loss"], test_acc=acc,
                  committee=[r for r, x in enumerate(st["roles"]) if x & 2])
    errs = eng.drain_blocks()
    summary = dict(rounds=a.rounds, wall_s=round(time.time() - t0, 3), timing=timer.summary(),
                   ledger_mismatches=errs, chain_ok=eng.host_ledger.verify_chain(),
                   blocks=eng.host_ledger.n_blocks(), symm=eng.heap.describe())
    if a.checkpoint:
        from .utils.checkpoint import save_checkpoint
        summary["checkpoint"] = save_checkpoint(a.checkpoint, eng)
    if rank == 0:
        print("SUMMARY " + json.dumps(summary))
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


def run_multiclient(a):
    """--clients N on one GPU: N virtual clients, the committee protocol in one captured graph."""
    from .engine.multiclient import MultiClientEngine
    if a.model != "mlp":
        raise SystemExit("--clients runs the MLP only")
    S, B, LR = a.samples or 4096, a.batch or 512, a.lr or (0.002 if a.optimizer == "adam" else 0.05)
    cfg = FLConfig(clients=a.clients, committee_size=a.committee, needed_updates=a.needed,
                   aggregate_count=a.aggregate, batch_size=B, samples_per_client=S, learning_rate=LR,
                   optimizer=a.optimizer, byzantine_ranks=a.byzantine, ring_slots=1024,
                   dtype=a.dtype, non_iid_alpha=a.alpha, **a.fedopt).validate()
    # shard sizes in whole batches (every client trains at least one; fp8 batches are 128-row tiles)
    sizes = client_sizes(a.clients, S, sigma=a.size_sigma, multiple=B, seed=7) if a.size_sigma > 0 else None
    shards = femnist_like(a.clients, S, seed=7, alpha=cfg.non_iid_alpha, sizes=sizes)
    test = femnist_like(1, 2048, seed=7, only=0)[0]
    eng = MultiClientEngine(cfg, shards, device=0)
    print(f"[clients] alpha {cfg.non_iid_alpha} size_sigma {a.size_sigma} rows per client "
          f"{eng.rows_per_client}")
    print(f"[clients] prox_mu {cfg.prox_mu} server_optimizer {cfg.server_optimizer} server_lr {cfg.server_lr} "
          f"server_beta1 {cfg.server_beta1} server_beta2 {cfg.server_beta2} server_tau {cfg.server_tau}")
    eng.capture()
    log = RunLog(rank=0)
    timer = PhaseTimer()
    t0 = time.time()
    for _ in range(a.rounds):
        with timer.phase("round"):
            eng.run_round()
        st = eng.read_state()
        log.round(st["epoch"] - 1, st["global_loss"], test_acc=eng.evaluate(test),
                  committee=[r for r, x in enumerate(st["roles"]) if x & 2])
    errs = eng.drain_blocks()
    summary = dict(rounds=a.rounds, clients=a.clients, alpha=cfg.non_iid_alpha, size_sigma=a.size_sigma,
                   rows_per_client=eng.rows_per_client, prox_mu=cfg.prox_mu,
                   server_optimizer=cfg.server_optimizer, server_lr=cfg.server_lr, server_beta1=cfg.server_beta1,
                   server_beta2=cfg.server_beta2, server_tau=cfg.server_tau, wall_s=round(time.time() - t0, 3),
                   timing=timer.summary(), ledger_mismatches=errs, chain_ok=eng.host_ledger.verify_chain(),
                   blocks=eng.host_ledger.n_blocks(), launches_per_round=eng.launches_per_round)
    print("SUMMARY " + json.dumps(summary))


if __name__ == "__main__":
    main()
