"""Rounds/s of the multi-client engine (engine/multiclient.py) on one GPU.

    python scripts/bench_multiclient.py [--clients 8 20 32] [--skewed 20] [--size-sigma 0.8]
                                        [--fedopt 20] [--repeat 1] [--steps 20] [--warmup 5]

For C clients (committee / needed / aggregate in the reference's 20 / 4 / 10 / 6 proportions),
4096 samples and batch 512 per client, fp8 + Adam and bf16 + SGD: device-event time of the
captured round graph with an L2 flush between timed rounds (as bench.py), the split into
training / validation / consensus + FedAvg (the same round captured as three graphs), and FedAvg
alone against the HBM roofline.  Prints one JSON line per configuration.

``--skewed C``: the same C-client workload with unequal shards -- log-normal sizes
(``client_sizes``, ``--size-sigma``) in whole batches with the same total sample count (C x 4096),
so training time is comparable; the validation grid spans the largest member's rows.

``--fedopt C``: the equal-shard C-client workload with FedProx clients (prox_mu 0.01) and a FedAdam
server (server_optimizer adam), to compare its train / validate / consensus + FedAvg split row
against row with the plain rows.  ``--repeat N`` runs the whole list N times, interleaved, which
shows the run-to-run spread.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from bflc_demo_b200.config import FLConfig  # noqa: E402
from bflc_demo_b200.data.synthetic import client_sizes, femnist_like  # noqa: E402
from bflc_demo_b200.engine.multiclient import MultiClientEngine  # noqa: E402

HBM_PEAK = 7.7e12   # HBM3e bandwidth of one HGX B200 GPU, bytes/s (NVIDIA data sheet)


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=20)
        return out.stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def timed(fn, flush, reps, stream):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            flush.zero_()
            a.record(stream)
            fn()
            b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


FEDOPT = dict(prox_mu=0.01, server_optimizer="adam", server_lr=0.01)


def bench(clients, dtype, opt, steps, warmup, flush, size_sigma=0.0, fedopt=None):
    cfg = FLConfig.reference_scaled(clients, model="mlp", dataset="femnist", hidden=256, batch_size=512,
                                    samples_per_client=4096, dtype=dtype, optimizer=opt,
                                    learning_rate=0.002 if opt == "adam" else 0.05, ring_slots=1024,
                                    **(fedopt or {}))
    sizes = client_sizes(clients, 4096, sigma=size_sigma, multiple=512, seed=7) if size_sigma > 0 else None
    eng = MultiClientEngine(cfg, femnist_like(clients, 4096, seed=7, sizes=sizes), device=0)
    eng.capture()
    for _ in range(warmup):
        eng.run_round()
    torch.cuda.synchronize()
    s = eng.stream
    round_us = timed(lambda: eng.run_round(), flush, steps, s)
    # per-phase graphs (the same round, split in three)
    graphs = []
    for ph in (eng.phase_train, eng.phase_validate, eng.phase_aggregate):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            ph()
        graphs.append(g)
    split = [0.0, 0.0, 0.0]
    for _ in range(steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.stream(s):
            flush.zero_()
            ev[0].record(s)
            for i, g in enumerate(graphs):
                g.replay()
                ev[i + 1].record(s)
        ev[3].synchronize()
        for i in range(3):
            split[i] += ev[i].elapsed_time(ev[i + 1]) * 1e3 / steps
    errs = eng.drain_blocks()
    st = eng.read_state()
    n_sel = bin(st["selected_mask"]).count("1")
    # FedAvg alone (last: it re-averages the already averaged masters, the ledger is not drained again)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        eng.fedavg()
    with torch.cuda.stream(s):
        g.replay()
    fedavg_us = timed(lambda: g.replay(), flush, steps, s)
    P = eng.n_params
    fed_bytes = n_sel * P * 4 + P * 6 + clients * P * 6
    # server optimizer: reads the current global model, reads and writes m (and v)
    fed_bytes += {"none": 0, "momentum": 3, "adam": 5, "yogi": 5}[cfg.server_optimizer] * P * 4
    rows = eng.rows_per_client
    return dict(clients=clients, committee=cfg.committee_size, needed=cfg.needed_updates,
                aggregate=cfg.aggregate_count, dtype=dtype, optimizer=opt, samples=4096, batch=512,
                size_sigma=size_sigma, prox_mu=cfg.prox_mu, server_optimizer=cfg.server_optimizer,
                samples_total=sum(rows), rows_min=min(rows), rows_max=max(rows),
                round_us=round(round_us, 1), rounds_per_s=round(1e6 / round_us, 1),
                train_us=round(split[0], 1), validate_us=round(split[1], 1),
                consensus_fedavg_us=round(split[2], 1), fedavg_us=round(fedavg_us, 1),
                fedavg_bytes=fed_bytes, fedavg_hbm_share=round(fed_bytes / (fedavg_us * 1e-6) / HBM_PEAK, 3),
                launches_per_round=eng.launches_per_round, ledger_mismatches=errs, epoch=st["epoch"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clients", type=int, nargs="*", default=[8, 20, 32])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--skewed", type=int, nargs="*", default=[20],
                    help="client counts also run with unequal shards (--size-sigma)")
    ap.add_argument("--size-sigma", type=float, default=0.8)
    ap.add_argument("--fedopt", type=int, nargs="*", default=[20],
                    help="client counts also run with FedProx + FedAdam (%s)" % FEDOPT)
    ap.add_argument("--repeat", type=int, default=1, help="run the whole list this many times")
    a = ap.parse_args()
    print(json.dumps(dict(gpu=torch.cuda.get_device_name(0), power_limit=power_limit(),
                          hbm_peak_bytes_per_s=HBM_PEAK)), flush=True)
    flush = torch.empty(256 << 20, device="cuda", dtype=torch.uint8)   # > L2
    runs = ([(c, 0.0, None) for c in a.clients] + [(c, a.size_sigma, None) for c in a.skewed] +
            [(c, 0.0, FEDOPT) for c in a.fedopt])
    for _ in range(a.repeat):
        for c, sigma, fo in runs:
            for dtype, opt in (("fp8", "adam"), ("bf16", "sgd")):
                print(json.dumps(bench(c, dtype, opt, a.steps, a.warmup, flush, sigma, fo)), flush=True)
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
