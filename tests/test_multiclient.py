"""Multi-client engine (engine/multiclient.py): the committee protocol with up to 32 clients on one
GPU.  The ledger test runs on the CPU; everything else needs a B200."""
import numpy as np
import pytest
import torch

from bflc_demo_b200._native import ledger as _ledger
from bflc_demo_b200.protocol import oracle as O

ROLE_TRAINER, ROLE_COMM = 1, 2


def _device_round_20(rng):
    """A 20-client device round: committee 0-3, 16 trainers, 10 admitted, top 6 aggregated."""
    n, comm, agg, needed = 20, 4, 6, 10
    roles = [ROLE_COMM if c < comm else ROLE_TRAINER for c in range(n)]
    trainers = [c for c in range(n) if roles[c] == ROLE_TRAINER]
    admitted = sorted(rng.choice(trainers, size=needed, replace=False).tolist())
    scores = {c: {t: float(np.float32(rng.integers(0, 512) / 512)) for t in admitted} for c in range(comm)}
    n_samples = {c: 4096 for c in range(n)}
    avg_cost = {c: float(np.float32(rng.uniform(0.5, 4.0))) for c in range(n)}
    ref = O.run_consensus(n, comm, agg, {c: roles[c] for c in range(n)}, admitted, scores, n_samples, avg_cost)
    rows = [[scores[c][t] if (c in scores and t in scores[c]) else 0.0 for t in range(n)] for c in range(n)]
    scored = [sum(1 << t for t in admitted) if c < comm else 0 for c in range(n)]
    rec = dict(epoch=0, role_before=roles, role_after=[ref.role_after[c] for c in range(n)], score_rows=rows,
               scored_mask=scored, n_samples=[n_samples[c] for c in range(n)],
               avg_cost=[avg_cost[c] for c in range(n)], admitted_mask=sum(1 << t for t in admitted),
               selected_mask=sum(1 << t for t in ref.selected), global_loss=ref.global_loss,
               model_digest=0x1234, weight_by_score=0)
    return roles, rec, ref


def _ledger_20():
    L = _ledger()
    c = L.LedgerConfig()
    c.client_num, c.comm_count, c.aggregate_count, c.needed_update_count = 20, 4, 6, 10
    c.model_size, c.learning_rate = 16, 0.001
    return L.Ledger(c)


def test_host_ledger_accepts_a_20_client_device_round():
    rng = np.random.default_rng(11)
    roles, rec, ref = _device_round_20(rng)
    led = _ledger_20()
    led.Bootstrap(roles)
    assert led.AppendDeviceRound(rec) == ""
    blk = led.blocks()[-1]
    assert blk["selected"] == ref.selected and len(blk["admitted"]) == 10 and len(blk["committee"]) == 4
    assert led.verify_chain() and led.epoch() == 1
    # the same record with one bit of the selected mask flipped is refused
    led2 = _ledger_20()
    led2.Bootstrap(roles)
    bad = dict(rec)
    flip = next(t for t in range(20) if (rec["admitted_mask"] >> t) & 1 and not (rec["selected_mask"] >> t) & 1)
    bad["selected_mask"] = rec["selected_mask"] ^ (1 << flip)
    assert led2.AppendDeviceRound(bad) == "selected set mismatch"
    assert led2.epoch() == 0


# ---------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu
needs_cuda = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")


def _engine(dtype="fp8", optimizer="adam", clients=20, samples=1024, batch=256, val=512, lr=None, noise=48.0,
            **kw):
    from bflc_demo_b200.config import FLConfig
    from bflc_demo_b200.data.synthetic import femnist_like
    from bflc_demo_b200.engine.multiclient import MultiClientEngine
    cfg = FLConfig(clients=clients, committee_size=4, needed_updates=10, aggregate_count=6, hidden=256,
                   batch_size=batch, samples_per_client=samples, val_samples=val, dtype=dtype,
                   optimizer=optimizer, learning_rate=lr or (0.002 if optimizer == "adam" else 0.05),
                   ring_slots=64, **kw).validate()
    shards = femnist_like(clients, samples, seed=7, noise=noise)
    return MultiClientEngine(cfg, shards, device=0), shards


def _test_shard(noise=48.0):
    from bflc_demo_b200.data.synthetic import femnist_like
    return femnist_like(1, 2048, seed=7, only=0, noise=noise)[0]


@gpu
@needs_cuda
def test_reference_protocol_20_clients_fp8_adam():
    eng, _ = _engine("fp8", "adam")
    test = _test_shard()
    acc0 = eng.evaluate(test)
    eng.capture()
    committees = set()
    for _ in range(8):
        eng.run_round()
        committees.add(tuple(eng.committee()))
    assert eng.drain_blocks() == []
    assert eng.host_ledger.verify_chain() and eng.host_ledger.n_blocks() == 9
    for blk in eng.host_ledger.blocks():
        assert len(blk["committee"]) == 4
        assert len(blk["admitted"]) == 10 and len(blk["selected"]) == 6
        assert abs(sum(blk["weight"]) - 1.0) < 1e-5
    assert len(committees) > 1, "the committee never changed"
    acc = eng.evaluate(test)
    print(f"[multiclient] 20 clients fp8+adam: acc {acc0:.3f} -> {acc:.3f}, "
          f"launches/round {eng.launches_per_round}")
    assert acc > acc0 + 0.2


@gpu
@needs_cuda
@pytest.mark.parametrize("dtype", ["bf16", "fp8"])
def test_fedavg_is_bit_exact(dtype):
    eng, _ = _engine(dtype, "sgd" if dtype == "bf16" else "adam")
    worst = 0.0
    for _ in range(3):
        eng.phase_train()
        eng.phase_validate()
        masters = eng.master.clone()
        eng.phase_aggregate()
        torch.cuda.synchronize()
        assert eng.drain_blocks() == []
        blk = eng.host_ledger.blocks()[-1]
        ref = torch.zeros(eng.n_params, device="cuda", dtype=torch.float64)
        for t, w in zip(blk["selected"], blk["weight"]):
            # fp32 fma(w, v, acc): the product is exact in fp64, one rounding back to fp32
            ref = (ref + masters[t].double() * float(np.float32(w))).float().double()
        got = eng.global_master.double()
        worst = max(worst, ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item())
        assert bool((got == ref).all()), f"{dtype}: FedAvg differs, worst rel err {worst:.3e}"
        for c in range(eng.cfg.clients):   # every client starts the next round from the new model
            assert torch.equal(eng.master[c], eng.global_master)
    print(f"[multiclient] FedAvg {dtype}: bit exact, worst relative error {worst:.3e}")


@gpu
@needs_cuda
def test_client_training_is_isolated():
    from bflc_demo_b200.models.mlp import FlatMLP
    eng, shards = _engine("fp8", "adam")
    g = eng.global_master.clone()
    eng.phase_train()
    torch.cuda.synchronize()
    for c in eng.trainers_now()[:3] + [eng.trainers_now()[-1]]:
        P = eng.n_params
        master, shadow = g.clone(), g.to(torch.bfloat16)
        grad = torch.zeros(P, device="cuda")
        tr = FlatMLP(eng.spec, master, shadow, grad, eng.cfg.batch_size, optimizer="adam",
                     lr=eng.cfg.learning_rate, fp8=True)
        tr.quantize_weights()
        bar = torch.zeros(1, device="cuda", dtype=torch.int32)
        tr.train_epoch_fused(eng.x_bf[c], eng.y[c], eng.steps, bar.data_ptr(), x_q=eng.x_q[c], x_sf=eng.x_sf[c])
        torch.cuda.synchronize()
        d = (eng.master[c] - master).abs().max().item()
        assert d < 2e-3 * max(master.abs().max().item(), 1.0), (c, d)
        assert (eng.master[c] - g).abs().max().item() > 10 * d   # it did train


def _reference_correct(eng):
    """correct[member][candidate] from the one-client-per-GPU validation kernel (mlp_val), launched
    per committee member over <= 8 candidates at a time, reading the same candidate buffers."""
    m, e = eng.mod, eng.spec.by_name
    plan = eng.plan_bytes.cpu().numpy().view(np.int32)
    sz = eng.sz
    n_cand = int(plan[sz["mc_plan_n_cand_off"] // 4])
    cands = [int(x) for x in plan[sz["mc_plan_cand_off"] // 4:][:n_cand]]
    n_comm = int(plan[sz["mc_plan_n_comm_off"] // 4])
    members = [int(x) for x in plan[sz["mc_plan_comm_off"] // 4:][:n_comm]]
    out = np.zeros((32, 32), dtype=np.int64)
    for mem in members:
        for g0 in range(0, n_cand, 8):
            grp = cands[g0:g0 + 8]
            d1 = m.gemm_dynamic_bytes(len(grp), grp, [eng.master[t].data_ptr() + 4 * e["b1"].offset for t in grp])
            d2 = m.gemm_dynamic_bytes(len(grp), [32 + t for t in grp],
                                      [eng.master[t].data_ptr() + 4 * e["b2"].offset for t in grp])
            dyn = torch.frombuffer(bytearray(d1 + d2), dtype=torch.uint8).cuda()
            corr = torch.zeros(8, device="cuda", dtype=torch.int32)
            xs = (eng.x_q if eng.fp8 else eng.x_bf)[mem][:eng.n_val]
            if eng.fp8:
                blobs = torch.tensor([eng.trainers[t].work_q.data_ptr() for t in grp], dtype=torch.int64).cuda()
                m.mlp_val(xs, eng.y[mem][:eng.n_val], corr, eng.w_maps, dyn.data_ptr(), dyn.data_ptr() + len(d1),
                          eng.n_val, eng.in_dim, 256, eng.n_classes, len(grp), eng.x_sf[mem], blobs.data_ptr())
            else:
                m.mlp_val(xs, eng.y[mem][:eng.n_val], corr, eng.w_maps, dyn.data_ptr(), dyn.data_ptr() + len(d1),
                          eng.n_val, eng.in_dim, 256, eng.n_classes, len(grp))
            torch.cuda.synchronize()
            for z, t in enumerate(grp):
                out[mem, t] = int(corr[z].item())
    return out, members, cands


@gpu
@needs_cuda
@pytest.mark.parametrize("dtype", ["bf16", "fp8"])
def test_validation_matches_single_client_kernel(dtype):
    eng, _ = _engine(dtype, "sgd")
    for _ in range(2):
        eng.phase_train()
        eng.phase_validate()
        torch.cuda.synchronize()
        got = eng.correct.cpu().numpy().astype(np.int64)
        ref, members, cands = _reference_correct(eng)
        assert len(members) == 4 and len(cands) == 10
        for mem in members:
            for t in cands:
                assert got[mem, t] == ref[mem, t], (mem, t, got[mem, t], ref[mem, t])
                assert got[mem, t] > 0
        eng.phase_aggregate()


@gpu
@needs_cuda
def test_score_filter_rejects_byzantine_clients():
    # a noisy task the model does not saturate within the run: once every update scores 100 %, a
    # scaled-back step cannot be told apart by accuracy any more
    eng, _ = _engine("fp8", "adam", byzantine_ranks=[5, 11], byzantine_scale=5.0, noise=400.0, lr=0.001)
    test = _test_shard(noise=400.0)
    acc0 = eng.evaluate(test)
    assert eng.committee() == [0, 1, 2, 3]
    eng.capture()
    for _ in range(7):
        eng.run_round()
    assert eng.drain_blocks() == []
    admitted = {5: 0, 11: 0}
    for blk in eng.host_ledger.blocks():
        for b in (5, 11):
            assert b not in blk["selected"], blk
            assert b not in blk["committee"], blk
            admitted[b] += b in blk["admitted"]
    assert admitted[5] > 0 and admitted[11] > 0, admitted
    acc = eng.evaluate(test)
    print(f"[multiclient] Byzantine 5, 11 admitted {admitted}, never selected; acc {acc0:.3f} -> {acc:.3f}")
    assert acc > acc0 + 0.1
