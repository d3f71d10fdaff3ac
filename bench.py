#!/usr/bin/env python
"""Headline benchmark: federated rounds/sec of the committee-consensus protocol on a 2-layer
MLP over synthetic FEMNIST (BASELINE.json), one client per B200.

  python bench.py --gpus N --steps K --warmup W            # fused engine (the product)
  python bench.py --impl nccl ...                          # OUR NCCL+cuBLAS baseline arm
  python bench.py --impl reference ...                     # the unmodified reference (cannot
                                                           # be installed here -> "unavailable")

A "step" is one full federated round: every trainer runs one local pass (steps x batch
samples, forward+backward+optimizer), uploads; every committee member validates every
candidate on its own shard; median / top-K / sample-weighted FedAvg; re-election.
Per-GPU work is fixed as N grows (weak scaling).

Timing: W >= 3 untimed rounds, then K rounds each bracketed by CUDA events on the launching
stream; between timed rounds a 256 MiB buffer is written to flush the 126 MB L2 and the
ranks re-synchronise (barrier + cudaDeviceSynchronize) OUTSIDE the timed interval; the
per-round time is the max over ranks and the reported time is the sum over the K rounds.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

REFERENCE_UNAVAILABLE = (
    "reference is a FISCO-BCOS precompiled contract + TF1 client with no setup.py/pyproject and "
    "no GPU code; pip install of /root/reference fails (not a Python project) and it needs "
    "FISCO-BCOS 2.x, nlohmann/json, the FISCO python-sdk, solc and TensorFlow, none available "
    "offline (see DESIGN.md 'Reference arm')")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="fused", choices=["fused", "nccl", "reference"])
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--samples", type=int, default=4096, help="samples per client per round")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--optimizer", default="adam", choices=["sgd", "adam"])
    ap.add_argument("--dtype", default="fp8", choices=["fp8", "bf16"],
                    help="fp8 = block-scaled fp8 (MXFP8) forward GEMMs, BASELINE.json config #2")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--no-fused-step", action="store_true", help="fused arm: one launch per GEMM instead of the persistent training kernel")
    ap.add_argument("--no-stage", action="store_true", help="fused arm: validation GEMMs TMA-load peers' HBM directly")
    ap.add_argument("--broadcast", action="store_true", help="nccl arm: literal average+broadcast")
    ap.add_argument("--no-baseline", action="store_true",
                    help="fused arm: skip timing our NCCL+cuBLAS baseline in the same process (vs_baseline = null)")
    ap.add_argument("--two-shot", default="auto", choices=["auto", "on", "off"],
                    help="fused arm: FedAvg as reduce-own-slice + multicast publish (auto: by model size)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed round computed (global model + round result) "
                         "as DIR/<name>.npy; the inputs are seeded, so two builds compare output for output")
    return ap.parse_args()


DUMP_MAX_ELEMS = 1 << 21     # per array (8 MB of fp32): a dump of the MLP's four tensors stays < 64 MB


def round_outputs(eng) -> dict:
    """What a caller of the timed round receives: the global model (fp32, per tensor) and the
    round's result (epoch, roles, global loss; the fused engine's ledger page adds the committee's
    median scores and the FedAvg selection mask).  An array above DUMP_MAX_ELEMS is replaced by a
    fixed, seeded sample of its elements."""
    import numpy as np

    if hasattr(eng, "global_master"):          # FusedEngine: replicated ledger page on the device
        st = eng.read_state()
        model = eng.spec.views(eng.global_master)
        res = dict(epoch=st["epoch"], roles=st["roles"], median_scores=st["median"],
                   selected_mask=st["selected_mask"], global_loss=st["global_loss"])
    else:                                      # NcclBaselineEngine: host copy of the round's result
        model = eng.spec.views(eng.global_w)
        res = dict(epoch=eng.epoch, roles=eng.roles, global_loss=eng.global_loss)
    out = {f"global_{k}": v.detach().float().cpu().numpy() for k, v in model.items()}
    out.update({k: np.atleast_1d(np.asarray(v, dtype=np.float64)) for k, v in res.items()})
    for k, a in out.items():
        if a.size > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            out[k] = a.reshape(-1)[idx]
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.proc = None
        self.path = f"/tmp/bflc_clocks_{os.getpid()}.csv"
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def main():
    args = parse()
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:      # one line even when launched under torchrun
            print(json.dumps({"impl": "reference", "unavailable": REFERENCE_UNAVAILABLE}))
        return 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: re-launch ourselves under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
               f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1", "--master-port",
               os.environ.get("MASTER_PORT", "29531"), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n = max(world, 1)
    assert n == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    import torch
    import torch.distributed as dist

    from bflc_demo_b200.config import FLConfig
    from bflc_demo_b200.data.synthetic import femnist_like

    torch.cuda.set_device(local_rank)
    group = None
    if n > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = FLConfig.for_world(n, model="mlp", dataset="femnist", hidden=args.hidden,
                             batch_size=args.batch, samples_per_client=args.samples,
                             optimizer=args.optimizer,
                             learning_rate=0.05 if args.optimizer == "sgd" else 1e-3, dtype=args.dtype,
                             cuda_graph=not args.no_graph, ring_slots=1024,
                             fused_step=not args.no_fused_step, stage_candidates=not args.no_stage,
                             two_shot={"auto": None, "on": True, "off": False}[args.two_shot])
    shard = femnist_like(n, args.samples, seed=7, only=rank)[0]
    # a small pool of distinct pinned input sets the e2e loop cycles through
    pool = [femnist_like(n, args.samples, seed=100 + i, only=rank)[0] for i in range(3)]

    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    _start = torch.zeros(1, dtype=torch.int64, device="cuda") if n > 1 else None
    _ALIGN = os.environ.get("BFLC_BENCH_ALIGN", "1") != "0"

    def sync_all():
        """Barrier + synchronize on every rank; then the ranks leave together.  An NCCL barrier
        releases the processes several (up to ~20) microseconds apart, and with a step of ~250 us
        that host-side skew lands 1:1 in the max-over-ranks time of whoever started first (it waits
        for the late ranks' uploads).  All ranks run on one node, so CLOCK_MONOTONIC is common: agree
        on an instant a little in the future and spin until it -- outside every timed interval."""
        torch.cuda.synchronize()
        if n > 1:
            dist.barrier()
            if not _ALIGN:
                torch.cuda.synchronize()
                return
            _start[0] = time.monotonic_ns() + 300_000
            dist.all_reduce(_start, op=dist.ReduceOp.MAX)
            tgt = int(_start.item())          # (also synchronizes the device)
            while time.monotonic_ns() < tgt:
                pass

    def reduce_max(vals):
        t = torch.tensor(vals, device="cuda", dtype=torch.float64)
        if n > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def measure(eng, drain, want_clocks, dump=False):
        """W warm-up rounds, then K device-timed rounds (resident inputs), K e2e rounds (pinned
        host inputs in, result out, inside the timed interval) and K back-to-back rounds.
        Every timed round: CUDA events on the engine stream, L2 flush + barrier outside the
        interval, max over ranks.  ``dump``: also return round_outputs() of the K-th device-timed
        round (read after it, outside every timed interval)."""
        pool_x = [p.x.reshape(len(p), -1).contiguous().pin_memory() for p in pool]
        ydt = eng.host_y.dtype
        pool_y = [p.y.to(ydt).contiguous().pin_memory() for p in pool]

        def timed(fn, k):
            out = []
            for i in range(k):
                if flush is not None:
                    flush.fill_(i & 0xFF)
                sync_all()
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record(eng.stream)      # (no stream context manager: its Python cost would sit
                fn(i)                      #  between the event and the launch, inside the interval)
                e1.record(eng.stream)
                e1.synchronize()
                out.append(e0.elapsed_time(e1))
            return out

        def round_only(i):
            eng.run_round()

        def round_e2e(i):
            eng.run_round_e2e(pool_x[i % len(pool_x)], pool_y[i % len(pool_y)])

        for i in range(W):
            round_e2e(i)
        if n > 1:
            # a few more untimed rounds through the exact timed paths (barrier, flush, events) so
            # that every rank's launch path is warm before the first timed round: the first
            # multi-GPU run on a fresh box otherwise shows the ranks' launches further apart
            timed(round_only, 8)
            timed(round_e2e, 4)
        sync_all()
        sampler = ClockSampler(local_rank) if (rank == 0 and want_clocks) else None
        if sampler:
            sampler.start()
        launches0 = _launch_count()
        errs = list(drain())
        t_dev = timed(round_only, args.steps)
        errs += drain()
        launches = _launch_count() - launches0
        outputs = None
        if dump:
            sync_all()          # every rank's round, peers' writes into this heap included, has landed
            outputs = round_outputs(eng)
        t_e2e = timed(round_e2e, args.steps)
        errs += drain()
        sync_all()   # back-to-back (no flush, no per-round barrier) for context
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(eng.stream):
            e0.record()
        for i in range(args.steps):
            eng.run_round()
        with torch.cuda.stream(eng.stream):
            e1.record()
        e1.synchronize()
        pipelined_ms = e0.elapsed_time(e1) / args.steps
        sync_all()
        clocks = sampler.stop() if sampler else None
        errs += drain()
        return dict(dev_ms=sum(reduce_max(t_dev)), e2e_ms=sum(reduce_max(t_e2e)),
                    pipe_ms=reduce_max([pipelined_ms])[0], launches=int(launches), clocks=clocks,
                    ledger_errs=errs, outputs=outputs)

    W = max(args.warmup, 3)
    base = None
    if args.impl == "fused" and not args.no_baseline:
        # The comparator, timed by THIS invocation with the same N / K / W and the same timing
        # code: OUR NCCL + cuBLAS build of the same round (the reference cannot be installed --
        # see --impl reference).  bf16 cuBLAS GEMMs: the library path a PyTorch user has.
        from bflc_demo_b200.engine.nccl_baseline import NcclBaselineEngine
        beng = NcclBaselineEngine(cfg, shard, rank=rank, world=n, device=local_rank, group=group)
        beng.capture()
        bm = measure(beng, lambda: [], False)
        base = {"impl": "nccl+cublas baseline (ours: torch ops, cuBLASLt epilogues, NCCL all_gather, "
                        "device-side election, one CUDA graph per role; NOT a reference build)",
                "dtype": "bf16", "graph_captured": bool(beng.graphs),
                "value": args.steps / (bm["dev_ms"] / 1e3), "ms_per_step": bm["dev_ms"] / args.steps,
                "e2e_value": args.steps / (bm["e2e_ms"] / 1e3), "e2e_ms_per_step": bm["e2e_ms"] / args.steps,
                "pipelined_ms_per_step_no_flush": bm["pipe_ms"]}
        del beng
        torch.cuda.empty_cache()

    if args.impl == "fused":
        from bflc_demo_b200.engine.fused import FusedEngine
        eng = FusedEngine(cfg, shard, rank=rank, world=n, device=local_rank, group=group)
    else:
        from bflc_demo_b200.engine.nccl_baseline import NcclBaselineEngine
        eng = NcclBaselineEngine(cfg, shard, rank=rank, world=n, device=local_rank, group=group,
                                 broadcast=args.broadcast)
    eng.capture()
    drain = (lambda: eng.drain_blocks()) if args.impl == "fused" else (lambda: [])
    mres = measure(eng, drain, True, dump=args.dump_outputs is not None)
    dev_ms, e2e_ms, pipe_ms = mres["dev_ms"], mres["e2e_ms"], mres["pipe_ms"]
    clocks, launches, ledger_errs = mres["clocks"], mres["launches"], mres["ledger_errs"]

    # consistency: the fused engine's host ledger re-executes every device election
    extra = {}
    if args.impl == "fused":
        errs = ledger_errs + eng.drain_blocks()
        st = eng.read_state()
        extra = {"ledger_blocks": eng.host_ledger.n_blocks(), "ledger_mismatches": errs[:2],
                 "chain_ok": eng.host_ledger.verify_chain(), "epoch": st["epoch"],
                 "global_loss": st["global_loss"], "symm": eng.heap.describe(),
                 "launches_per_round": eng.launches_per_round, "fused_step": eng.fused_step,
                 "fused_upload": bool(eng.fused_upload), "two_shot": bool(eng.two_shot),
                 "e2e_input_pipeline": bool(getattr(eng, "pipelined_input", False)),
                 "staged_validation": eng.staged}
        # device-stamped phase breakdown (%globaltimer inside the fed kernels), median of 9 extra
        # rounds per rank, then the max over ranks of each phase
        samples = []
        for _ in range(9):
            sync_all()
            eng.run_round()
            samples.append(eng.read_stamps())
        drain()
        keys = sorted(samples[0])
        med = [sorted(s[k] for s in samples)[len(samples) // 2] for k in keys]
        ph = {k: round(v, 2) for k, v in zip(keys, reduce_max(med))}
        # BASELINE's second metric: the part of a round that is neither local training nor the
        # committee's validation GEMMs (upload + pull + score exchange + FedAvg + publish + skew)
        ph["exposed_comm_us"] = round(max(ph["round_us"] - ph["train_us"] - ph["validate_us"], 0.0), 2)
        extra["phases_us_max_over_ranks"] = ph
        # the same stamps for end-to-end rounds (inputs streamed from pinned host memory): the
        # difference to the e2e time per round is what happens before the first / after the last kernel
        samples = []
        for i in range(5):
            sync_all()
            eng.run_round_e2e()
            samples.append(eng.read_stamps())
        drain()
        med = [sorted(s[k] for s in samples)[len(samples) // 2] for k in keys]
        extra["phases_us_e2e_round"] = {k: round(v, 2) for k, v in zip(keys, reduce_max(med))}
        if n > 1:
            digs = [None] * n
            dist.all_gather_object(digs, st["model_digest"])
            extra["replicas_bit_identical"] = len(set(digs)) == 1
        gl = eng.launches_per_round * args.steps
    else:
        extra = {"epoch": eng.epoch, "global_loss": eng.global_loss,
                 "graph_captured": bool(getattr(eng, "graphs", None))}
        gl = int(launches)

    if rank == 0 and args.dump_outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in mres["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    if rank == 0:
        K = args.steps
        trainers = cfg.n_trainers
        line = {
            "metric": "federated_rounds_per_sec",
            "value": K / (dev_ms / 1e3),
            "unit": "rounds/s",
            "n_gpus": n, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K,
            "higher_is_better": True, "scaling": "weak",
            # BASELINE.md publishes no throughput and the reference cannot be installed (see --impl
            # reference); the comparator is OUR NCCL+cuBLAS build of the same round, timed by this
            # same invocation (key "baseline"): vs_baseline = value / baseline.value
            "vs_baseline": (K / (dev_ms / 1e3)) / base["value"] if base else None,
            "dtype": "mxfp8" if (args.dtype == "fp8" and args.impl == "fused") else "bf16", "data": "synthetic (class-conditional FEMNIST-like 28x28 uint8, 62 classes; random-init weights)",
            "impl": args.impl if args.impl == "fused" else "nccl-baseline (ours, not a reference build)",
            "config": {"model": f"mlp_784x{args.hidden}x62", "global_batch": trainers * eng.S,
                       "seq_len": None, "parallelism": f"fed-dp{n} (committee {cfg.committee_size}, "
                       f"trainers {trainers}, top-{cfg.aggregate_count})",
                       "samples_per_client_per_round": eng.S, "local_batch": args.batch,
                       "local_steps": eng.steps, "val_samples": eng.n_val,
                       "optimizer": args.optimizer, "cuda_graph": not args.no_graph,
                       "l2": "flushed between timed rounds (256 MiB write, outside the timed interval)"
                             if flush is not None else "not flushed",
                       "pipelined_ms_per_step_no_flush": pipe_ms},
            "clocks": clocks,
            "e2e": {"value": K / (e2e_ms / 1e3), "unit": "rounds/s", "ms_per_step": e2e_ms / K,
                    "h2d_bytes_per_step": eng.h2d_bytes_per_round,
                    "d2h_bytes_per_step": eng.d2h_bytes_per_round},
            "gpu_launches": gl,
            "baseline": dict(base, vs_baseline_e2e=(K / (e2e_ms / 1e3)) / base["e2e_value"]) if base else None,
            "extra": extra,
        }
        print(json.dumps(line))
    if n > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _launch_count() -> int:
    from bflc_demo_b200._native import C
    return int(C().launch_count())


if __name__ == "__main__":
    sys.exit(main())
