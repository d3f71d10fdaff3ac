"""Multi-client engine with unequal, non-IID shards: per-client sample counts, step counts and
validation rows, FedAvg weighted by each selected client's samples.  The data and ledger tests run
on the CPU; everything else needs a B200."""
import numpy as np
import pytest
import torch

from bflc_demo_b200._native import ledger as _ledger
from bflc_demo_b200.data.synthetic import client_sizes, femnist_like
from bflc_demo_b200.protocol import oracle as O

ROLE_TRAINER, ROLE_COMM = 1, 2

# 20 shards of 512..3072 rows (committee 0-3 at genesis).  fp8: multiples of 128; clients 7, 12, 17
# train 2 steps of 256 rows, clients 9, 16, 19 train 12.  bf16: members 1, 2 and 3 validate on a
# partial last tile, member 0 is larger than every other client (it sets the validation grid),
# member 1 (520 rows) is the smallest client (its extra CTAs exit).
FP8_SIZES = [3072, 512, 1024, 1536, 768, 2048, 1280, 512, 2560, 3072,
             1152, 1792, 512, 2304, 1408, 1024, 3072, 512, 1664, 3072]
BF16_SIZES = [3072, 520, 1000, 1300, 700, 2000, 1234, 640, 2500, 900,
              1100, 1800, 544, 2300, 1400, 1024, 2816, 777, 1666, 1900]


# ---------------------------------------------------------------------------------- CPU
def test_client_sizes_are_seeded_multiples():
    a = client_sizes(20, 1024, sigma=0.8, multiple=128, seed=3)
    assert a == client_sizes(20, 1024, sigma=0.8, multiple=128, seed=3)
    assert a != client_sizes(20, 1024, sigma=0.8, multiple=128, seed=4)
    assert len(a) == 20 and all(s > 0 and s % 128 == 0 for s in a)
    assert len(set(a)) > 1 and sum(a) == 20 * 1024
    assert client_sizes(20, 1024, sigma=0.0, multiple=128, seed=3) == [1024] * 20
    assert client_sizes(7, 300, sigma=0.0, multiple=128, seed=0) == [256] * 7
    # a very wide spread still gives every client at least one multiple
    b = client_sizes(32, 256, sigma=3.0, multiple=256, seed=1)
    assert min(b) == 256 and all(s % 256 == 0 for s in b)


def test_femnist_like_sizes_match_equal_shards():
    a = femnist_like(5, 384, seed=9, alpha=0.5)
    b = femnist_like(sizes=[384] * 5, seed=9, alpha=0.5)
    assert len(a) == len(b) == 5
    for s, t in zip(a, b):
        assert torch.equal(s.x, t.x) and torch.equal(s.y, t.y) and s.n_classes == t.n_classes
    c = femnist_like(sizes=[128, 640, 256], seed=9)
    assert [len(s) for s in c] == [128, 640, 256]
    # client i's shard depends only on (seed, i, sizes[i]), not on the other clients' sizes
    d = femnist_like(sizes=[999, 640], seed=9)
    assert torch.equal(c[1].x, d[1].x) and torch.equal(c[1].y, d[1].y)
    with pytest.raises(ValueError):
        femnist_like(3, sizes=[128, 256])


def test_host_ledger_weights_unequal_clients_by_samples():
    rng = np.random.default_rng(5)
    n, comm, agg, needed = 20, 4, 6, 10
    roles = [ROLE_COMM if c < comm else ROLE_TRAINER for c in range(n)]
    trainers = [c for c in range(n) if roles[c] == ROLE_TRAINER]
    admitted = sorted(rng.choice(trainers, size=needed, replace=False).tolist())
    n_val = {c: int(rng.integers(2, 25)) * 128 for c in range(comm)}
    scores = {c: {t: float(np.float32(rng.integers(0, n_val[c]) / n_val[c])) for t in admitted}
              for c in range(comm)}
    n_samples = {c: (0 if c < comm else int(rng.integers(2, 13)) * 256) for c in range(n)}
    avg_cost = {c: float(np.float32(rng.uniform(0.5, 4.0))) if c >= comm else 0.0 for c in range(n)}
    ref = O.run_consensus(n, comm, agg, {c: roles[c] for c in range(n)}, admitted, scores, n_samples, avg_cost)
    rows = [[scores[c][t] if (c in scores and t in scores[c]) else 0.0 for t in range(n)] for c in range(n)]
    rec = dict(epoch=0, role_before=roles, role_after=[ref.role_after[c] for c in range(n)], score_rows=rows,
               scored_mask=[sum(1 << t for t in admitted) if c < comm else 0 for c in range(n)],
               n_samples=[n_samples[c] for c in range(n)], avg_cost=[avg_cost[c] for c in range(n)],
               admitted_mask=sum(1 << t for t in admitted), selected_mask=sum(1 << t for t in ref.selected),
               global_loss=ref.global_loss, model_digest=0x77, weight_by_score=0)
    L = _ledger()
    cfg = L.LedgerConfig()
    cfg.client_num, cfg.comm_count, cfg.aggregate_count, cfg.needed_update_count = n, comm, agg, needed
    cfg.model_size, cfg.learning_rate = 16, 0.001
    led = L.Ledger(cfg)
    led.Bootstrap(roles)
    assert led.AppendDeviceRound(rec) == ""
    blk = led.blocks()[-1]
    sel = blk["selected"]
    assert sel == sorted(ref.selected) and len(sel) == agg
    total = sum(float(n_samples[t]) for t in sel)
    want = [float(np.float32(n_samples[t] / total)) for t in sel]
    assert blk["weight"] == want
    assert len(set(blk["weight"])) > 1, "the drawn sample counts should give unequal weights"
    assert led.verify_chain()


# ---------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu
needs_cuda = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")


def _engine(dtype="fp8", optimizer="adam", sizes=None, batch=256, val=0, lr=None, noise=48.0, alpha=0.0,
            **kw):
    from bflc_demo_b200.config import FLConfig
    from bflc_demo_b200.engine.multiclient import MultiClientEngine
    sizes = sizes or (FP8_SIZES if dtype == "fp8" else BF16_SIZES)
    cfg = FLConfig(clients=len(sizes), committee_size=4, needed_updates=10, aggregate_count=6, hidden=256,
                   batch_size=batch, samples_per_client=max(sizes), val_samples=val, dtype=dtype,
                   optimizer=optimizer, learning_rate=lr or (0.002 if optimizer == "adam" else 0.05),
                   ring_slots=64, non_iid_alpha=alpha, **kw).validate()
    shards = femnist_like(seed=7, noise=noise, alpha=alpha, sizes=sizes)
    return MultiClientEngine(cfg, shards, device=0), shards


def _test_shard(noise=48.0):
    return femnist_like(1, 2048, seed=7, only=0, noise=noise)[0]


def _check_weights(eng, blk):
    """Block weights are n_t / sum of the selected n, with n_t = S_t of that client."""
    S = eng.samples_per_client
    sel = blk["selected"]
    total = sum(float(S[t]) for t in sel)
    assert blk["weight"] == [float(np.float32(S[t] / total)) for t in sel], blk


@gpu
@needs_cuda
@pytest.mark.parametrize("dtype", ["fp8", "bf16"])
def test_unequal_clients_protocol(dtype):
    eng, _ = _engine(dtype, "adam" if dtype == "fp8" else "sgd")
    assert eng.steps is None and eng.n_val is None
    test = _test_shard()
    acc0 = eng.evaluate(test)
    eng.capture()
    for _ in range(8):
        eng.run_round()
    assert eng.drain_blocks() == []
    assert eng.host_ledger.verify_chain() and eng.host_ledger.n_blocks() == 9
    unequal = 0
    for blk in eng.host_ledger.blocks():
        assert len(blk["committee"]) == 4
        assert len(blk["admitted"]) == 10 and len(blk["selected"]) == 6
        _check_weights(eng, blk)
        unequal += len(set(blk["weight"])) > 1
    assert unequal > 0, "every block weighted its clients equally"
    acc = eng.evaluate(test)
    print(f"[hetero] 20 unequal clients {dtype}: acc {acc0:.3f} -> {acc:.3f}, blocks with unequal "
          f"weights {unequal}/9")
    assert acc > acc0 + 0.2


@gpu
@needs_cuda
@pytest.mark.parametrize("dtype", ["bf16", "fp8"])
def test_unequal_fedavg_is_bit_exact(dtype):
    eng, _ = _engine(dtype, "sgd" if dtype == "bf16" else "adam")
    unequal = 0
    for _ in range(3):
        eng.phase_train()
        eng.phase_validate()
        masters = eng.master.clone()
        eng.phase_aggregate()
        torch.cuda.synchronize()
        assert eng.drain_blocks() == []
        blk = eng.host_ledger.blocks()[-1]
        unequal += len(set(blk["weight"])) > 1
        ref = torch.zeros(eng.n_params, device="cuda", dtype=torch.float64)
        for t, w in zip(blk["selected"], blk["weight"]):
            # fp32 fma(w, v, acc): the product is exact in fp64, one rounding back to fp32
            ref = (ref + masters[t].double() * float(np.float32(w))).float().double()
        got = eng.global_master.double()
        assert bool((got == ref).all()), f"{dtype}: FedAvg with unequal weights differs"
        for c in range(eng.cfg.clients):
            assert torch.equal(eng.master[c], eng.global_master)
    assert unequal > 0


def _reference_correct(eng):
    """correct[member][candidate] from mlp_val, one launch per member and group of <= 8 candidates,
    on that member's own n_val_c rows."""
    m, e = eng.mod, eng.spec.by_name
    plan = eng.plan_bytes.cpu().numpy().view(np.int32)
    sz = eng.sz
    n_cand = int(plan[sz["mc_plan_n_cand_off"] // 4])
    cands = [int(x) for x in plan[sz["mc_plan_cand_off"] // 4:][:n_cand]]
    n_comm = int(plan[sz["mc_plan_n_comm_off"] // 4])
    members = [int(x) for x in plan[sz["mc_plan_comm_off"] // 4:][:n_comm]]
    out = np.zeros((32, 32), dtype=np.int64)
    for mem in members:
        nv = eng.n_val_per_client[mem]
        for g0 in range(0, n_cand, 8):
            grp = cands[g0:g0 + 8]
            d1 = m.gemm_dynamic_bytes(len(grp), grp, [eng.master[t].data_ptr() + 4 * e["b1"].offset for t in grp])
            d2 = m.gemm_dynamic_bytes(len(grp), [32 + t for t in grp],
                                      [eng.master[t].data_ptr() + 4 * e["b2"].offset for t in grp])
            dyn = torch.frombuffer(bytearray(d1 + d2), dtype=torch.uint8).cuda()
            corr = torch.zeros(8, device="cuda", dtype=torch.int32)
            xs = (eng.x_q if eng.fp8 else eng.x_bf)[mem][:nv]
            if eng.fp8:
                blobs = torch.tensor([eng.trainers[t].work_q.data_ptr() for t in grp], dtype=torch.int64).cuda()
                m.mlp_val(xs, eng.y[mem][:nv], corr, eng.w_maps, dyn.data_ptr(), dyn.data_ptr() + len(d1),
                          nv, eng.in_dim, 256, eng.n_classes, len(grp), eng.x_sf[mem], blobs.data_ptr())
            else:
                m.mlp_val(xs, eng.y[mem][:nv], corr, eng.w_maps, dyn.data_ptr(), dyn.data_ptr() + len(d1),
                          nv, eng.in_dim, 256, eng.n_classes, len(grp))
            torch.cuda.synchronize()
            for z, t in enumerate(grp):
                out[mem, t] = int(corr[z].item())
    return out, members, cands


@gpu
@needs_cuda
@pytest.mark.parametrize("dtype", ["bf16", "fp8"])
def test_validation_on_each_members_own_rows(dtype):
    eng, _ = _engine(dtype, "sgd")
    nv = eng.n_val_per_client
    assert nv[0] == max(nv) and nv[1] == min(nv)
    if dtype == "bf16":
        assert nv[0] > max(nv[1:]) and nv[2] % 128 and nv[3] % 128
    seen = set()
    for _ in range(3):
        eng.phase_train()
        eng.phase_validate()
        torch.cuda.synchronize()
        got = eng.correct.cpu().numpy().astype(np.int64)
        ref, members, cands = _reference_correct(eng)
        assert len(members) == 4 and len(cands) == 10
        seen.update(members)
        for mem in members:
            for t in cands:
                assert got[mem, t] == ref[mem, t], (mem, nv[mem], t, got[mem, t], ref[mem, t])
                assert 0 < got[mem, t] <= nv[mem]
        eng.phase_aggregate()
        assert eng.drain_blocks() == []
    assert {0, 1} <= seen     # the largest and the smallest member validated


def _ulp_dist(a, b):
    ia = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


@gpu
@needs_cuda
def test_scores_use_each_members_n_val():
    eng, _ = _engine("bf16", "sgd")
    for _ in range(3):
        eng.phase_train()
        eng.phase_validate()
        torch.cuda.synchronize()
        correct = eng.correct.cpu().numpy().astype(np.int64)
        eng.phase_aggregate()
        assert eng.drain_blocks() == []
        blk = eng.host_ledger.blocks()[-1]
        for i, mem in enumerate(blk["committee"]):
            for j, t in enumerate(blk["admitted"]):
                want = np.float32(correct[mem, t]) / np.float32(eng.n_val_per_client[mem])
                d = int(_ulp_dist(blk["scores"][i][j], want))
                assert d <= 2, (mem, t, blk["scores"][i][j], float(want), d)


def _plan_ints(eng, key, n):
    off = eng.sz[key] // 4
    return [int(x) for x in eng.plan_bytes.cpu().numpy().view(np.int32)[off:off + n]]


def _standalone(eng, c, g, m=None, v=None, base=0):
    """Client c's round from global model g with Adam moments (m, v) and step base `base`."""
    from bflc_demo_b200.models.mlp import FlatMLP
    P = eng.n_params
    master, shadow = g.clone(), g.to(torch.bfloat16)
    grad = torch.zeros(P, device="cuda")
    step = torch.tensor([base], device="cuda", dtype=torch.int32)
    tr = FlatMLP(eng.spec, master, shadow, grad, eng.cfg.batch_size, optimizer="adam",
                 lr=eng.cfg.learning_rate, step_dev_ptr=step.data_ptr(), fp8=True)
    if m is not None:
        tr.m.copy_(m)
        tr.v.copy_(v)
    tr.quantize_weights()
    bar = torch.zeros(1, device="cuda", dtype=torch.int32)
    tr.train_epoch_fused(eng.x_bf[c], eng.y[c], eng.steps_per_client[c], bar.data_ptr(),
                         x_q=eng.x_q[c], x_sf=eng.x_sf[c])
    torch.cuda.synchronize()
    return master


@gpu
@needs_cuda
def test_each_client_trains_its_own_steps():
    eng, _ = _engine("fp8", "adam")
    steps = eng.steps_per_client
    short, long_ = (7, 12, 17), (9, 16, 19)
    assert all(steps[c] == 2 for c in short) and all(steps[c] == 12 for c in long_)
    done = [0] * eng.cfg.clients
    for rnd in range(2):
        trainers = eng.trainers_now()
        picks = [next(c for c in short if c in trainers), next(c for c in long_ if c in trainers)]
        g = eng.global_master.clone()
        mv = {c: (eng.trainers[c].m.clone(), eng.trainers[c].v.clone()) for c in picks}
        eng.phase_train()
        torch.cuda.synchronize()
        # the Adam step base of every trainer is the sum of its own earlier step counts
        base = _plan_ints(eng, "mc_plan_opt_step_off", eng.cfg.clients)
        assert [base[c] for c in trainers] == [done[c] for c in trainers], (rnd, base, done)
        for c in picks:
            master = _standalone(eng, c, g, *mv[c], base=done[c])
            d = (eng.master[c] - master).abs().max().item()
            assert d < 2e-3 * max(master.abs().max().item(), 1.0), (rnd, c, steps[c], d)
            assert (eng.master[c] - g).abs().max().item() > 10 * d   # it did train
            if rnd == 1:
                # the same client with a wrong step base (a shared count) trains differently
                other = steps[picks[1]] if c == picks[0] else steps[picks[0]]
                wrong = _standalone(eng, c, g, *mv[c], base=other)
                assert (eng.master[c] - wrong).abs().max().item() > 4 * d, (c, "step base has no effect")
        for c in trainers:
            done[c] += steps[c]
        eng.phase_validate()
        eng.phase_aggregate()
        assert eng.drain_blocks() == []


@gpu
@needs_cuda
def test_score_filter_rejects_byzantine_client_with_largest_shard():
    sizes = [min(s, 2560) for s in FP8_SIZES]
    sizes[5] = 3072                          # client 5 holds the largest shard
    eng, _ = _engine("fp8", "adam", sizes=sizes, byzantine_ranks=[5, 11], byzantine_scale=5.0, noise=400.0,
                     lr=0.001)
    assert eng.samples_per_client[5] == max(eng.samples_per_client)
    test = _test_shard(noise=400.0)
    acc0 = eng.evaluate(test)
    assert eng.committee() == [0, 1, 2, 3]
    eng.capture()
    for _ in range(7):
        eng.run_round()
    assert eng.drain_blocks() == []
    admitted = {5: 0, 11: 0}
    for blk in eng.host_ledger.blocks():
        _check_weights(eng, blk)
        for b in (5, 11):
            assert b not in blk["selected"], blk
            assert b not in blk["committee"], blk
            admitted[b] += b in blk["admitted"]
    assert admitted[5] > 0 and admitted[11] > 0, admitted
    acc = eng.evaluate(test)
    print(f"[hetero] Byzantine 5 (largest shard), 11 admitted {admitted}, never selected; "
          f"acc {acc0:.3f} -> {acc:.3f}")
    assert acc > acc0 + 0.1


@gpu
@needs_cuda
def test_label_and_size_skew():
    sizes = client_sizes(20, 1536, sigma=0.8, multiple=256, seed=7)
    eng, _ = _engine("fp8", "adam", sizes=sizes, alpha=0.5)
    assert len(set(eng.rows_per_client)) > 1
    test = _test_shard()     # IID
    acc0 = eng.evaluate(test)
    eng.capture()
    for _ in range(8):
        eng.run_round()
    assert eng.drain_blocks() == []
    assert eng.host_ledger.verify_chain() and eng.host_ledger.n_blocks() == 9
    for blk in eng.host_ledger.blocks():
        _check_weights(eng, blk)
    acc = eng.evaluate(test)
    print(f"[hetero] alpha 0.5, sizes {min(sizes)}..{max(sizes)}: acc {acc0:.3f} -> {acc:.3f}")
    assert acc > acc0 + 0.1
