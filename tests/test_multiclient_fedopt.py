"""FedProx local training and server-side optimizers (FedAvgM, FedAdam, FedYogi) in the
multi-client engine.  Configuration, the other engines' refusal and the command line run on the
CPU; the kernels and the engine need a B200."""
import math

import numpy as np
import pytest
import torch

from bflc_demo_b200.config import FLConfig


# ---------------------------------------------------------------------------------- CPU
def test_config_defaults_are_plain_fedavg():
    c = FLConfig()
    assert c.prox_mu == 0.0 and c.server_optimizer == "none"
    assert (c.server_lr, c.server_beta1, c.server_beta2, c.server_tau) == (1.0, 0.9, 0.99, 1e-3)
    assert c.plain_fedavg
    c.require_plain_fedavg("any engine")


@pytest.mark.parametrize("field,value", [
    ("prox_mu", -0.1), ("prox_mu", math.inf), ("prox_mu", math.nan),
    ("server_optimizer", "sgd"), ("server_optimizer", ""),
    ("server_lr", 0.0), ("server_lr", -1.0),
    ("server_beta1", 1.0), ("server_beta1", -0.1), ("server_beta2", 1.0), ("server_beta2", -1e-9),
    ("server_tau", 0.0), ("server_tau", -1e-3)])
def test_config_rejects_invalid_values(field, value):
    with pytest.raises(ValueError, match=field):
        FLConfig(**{field: value}).validate()


def test_config_json_and_env_round_trip(monkeypatch):
    c = FLConfig(prox_mu=0.01, server_optimizer="yogi", server_lr=0.03, server_beta1=0.5,
                 server_beta2=0.9, server_tau=1e-4).validate()
    d = FLConfig.from_json(c.to_json())
    assert d == c and not d.plain_fedavg
    monkeypatch.setenv("BFLC_PROX_MU", "0.25")
    monkeypatch.setenv("BFLC_SERVER_OPTIMIZER", "momentum")
    e = FLConfig.from_env()
    assert e.prox_mu == 0.25 and e.server_optimizer == "momentum"
    monkeypatch.setenv("BFLC_SERVER_OPTIMIZER", "rmsprop")
    with pytest.raises(ValueError, match="server_optimizer"):
        FLConfig.from_env()


@pytest.mark.parametrize("kw", [dict(prox_mu=0.01), dict(server_optimizer="adam")])
def test_other_engines_refuse_fedprox_and_server_optimizers(kw):
    """The one-client-per-GPU engines implement neither: they refuse before any device work."""
    from bflc_demo_b200.data.synthetic import femnist_like
    from bflc_demo_b200.engine.fused import FusedEngine
    from bflc_demo_b200.engine.generic import GenericFedEngine
    from bflc_demo_b200.engine.nccl_baseline import NcclBaselineEngine
    cfg = FLConfig.for_world(1, hidden=256, batch_size=128, samples_per_client=512, **kw)
    shard = femnist_like(1, 512, seed=3)[0]
    for make in (lambda: FusedEngine(cfg, shard), lambda: GenericFedEngine(cfg, None, shard),
                 lambda: NcclBaselineEngine(cfg, shard)):
        with pytest.raises(ValueError, match="MultiClientEngine"):
            make()


def test_run_refuses_fedopt_flags_without_clients(capsys):
    from bflc_demo_b200 import run
    for argv in (["--prox-mu", "0.01"], ["--server-opt", "adam"], ["--server-lr", "0.1", "--clients", "1"]):
        with pytest.raises(SystemExit) as e:
            run.main(argv)
        assert e.value.code != 0
        assert "--clients" in capsys.readouterr().err


# ---------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu
needs_cuda = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")


def rel(x, ref):
    return ((x.float() - ref.float()).norm() / (ref.float().norm() + 1e-12)).item()


KEYS = ("w1", "b1", "w2", "b2")


def _train(spec, init, anchor, X, Y, xq, xsf, B, steps, opt, lr, mu, path, plan=-1, epiopt=-1):
    """Parameter deltas of one local pass: path "six" = per-GEMM launches + torch prox term,
    "bf16" / "fp8" = the persistent trainer."""
    from bflc_demo_b200.models.mlp import FlatMLP
    master = init.cuda().clone()
    tr = FlatMLP(spec, master, master.bfloat16(), torch.zeros_like(master), B, lr=lr, optimizer=opt,
                 fp8=path == "fp8", prox_mu=mu, prox_anchor=anchor if mu > 0 else None)
    if path == "six":
        tr.train_epoch(X, Y, steps)
    else:
        if path == "fp8":
            tr.quantize_weights()
        bar = torch.zeros(1, device="cuda", dtype=torch.int32)
        tr.train_epoch_fused(X, Y, steps, bar.data_ptr(), None, plan, epiopt,
                             x_q=xq if path == "fp8" else None, x_sf=xsf if path == "fp8" else None)
    torch.cuda.synchronize()
    assert float(tr.grad.abs().max()) == 0.0
    w0 = spec.views(init.cuda())
    return {k: v - w0[k] for k, v in spec.views(master).items()}, tr.loss_sum.item()


@gpu
@needs_cuda
@pytest.mark.parametrize("path,opt,plan,epiopt", [
    ("bf16", "sgd", -1, -1), ("bf16", "sgd", 0, 0), ("bf16", "sgd", 3, 1),
    ("bf16", "adam", -1, -1), ("bf16", "adam", 0, 0), ("bf16", "adam", 3, 1),
    ("fp8", "adam", -1, -1)])
def test_prox_term_in_the_persistent_trainer(path, opt, plan, epiopt):
    """The proximal term in all three update sites (E_OPT epilogue, bias CTA, flat P5 phase) vs the
    six-kernel path with the same term, and for SGD vs fp32 autograd of xent + mu/2 ||w - a||^2.
    The anchor is the initial model plus seeded noise, so the term is far from zero at step 1."""
    from bflc_demo_b200._native import C
    from bflc_demo_b200.models.mlp import mlp_spec, sf_bytes
    torch.manual_seed(13)
    B, steps, lr = (256, 3, 0.05) if opt == "sgd" else (512, 4, 1e-3)
    mu = 0.5
    spec = mlp_spec(784, 256, 62)
    init = torch.empty(spec.total)
    spec.init_(init, seed=2)
    anchor = (init + 0.1 * torch.randn(spec.total, generator=torch.Generator().manual_seed(5))).cuda()
    xu8 = (torch.rand(B * steps, 784, device="cuda") * 255).to(torch.uint8)
    Y = torch.randint(0, 62, (B * steps,), device="cuda", dtype=torch.int32)
    X = torch.empty(B * steps, 784, device="cuda", dtype=torch.bfloat16)
    xq = torch.zeros(B * steps, 784, device="cuda", dtype=torch.uint8)
    xsf = torch.full((sf_bytes(B * steps, 784),), 127, device="cuda", dtype=torch.uint8)
    C().prep_inputs(xu8, X, xq, xsf, 1.0 / 255.0)
    args = (spec, init, anchor, X, Y, xq, xsf, B, steps, opt, lr)
    got, loss = _train(*args, mu, path, plan, epiopt)
    ref, loss_ref = _train(*args, mu, "six")
    plain, loss_plain = _train(*args, 0.0, path, plan, epiopt)
    tol = 2e-2 if opt == "sgd" else 0.1          # the tolerances of the mu = 0 comparison
    for k in KEYS:
        assert rel(got[k], ref[k]) < tol, (k, rel(got[k], ref[k]))
        # a kernel that ignored mu would be this far off
        assert rel(plain[k], got[k]) > 10 * tol, (k, rel(plain[k], got[k]))
    # the reported loss is the cross-entropy alone, as the six-kernel path reports it
    assert abs(loss - loss_ref) / loss_ref < (2e-3 if path == "bf16" else 2e-2)
    if opt == "sgd":
        w0 = spec.views(init.cuda())
        a = spec.views(anchor)
        p = {k: v.clone().float() for k, v in w0.items()}
        for i in range(steps):
            xb, yb = X[i * B:(i + 1) * B].float(), Y[i * B:(i + 1) * B].long()
            q = {k: v.clone().requires_grad_(True) for k, v in p.items()}
            loss = torch.nn.functional.cross_entropy(
                torch.relu(xb @ q["w1"].t() + q["b1"]) @ q["w2"].t() + q["b2"], yb)
            loss = loss + mu / 2 * sum(((q[k] - a[k]) ** 2).sum() for k in KEYS)
            gr = torch.autograd.grad(loss, [q[k] for k in KEYS])
            p = {k: (q[k] - lr * g).detach() for k, g in zip(KEYS, gr)}
        for k in KEYS:
            assert rel(got[k], p[k] - w0[k]) < 6e-2, (k, rel(got[k], p[k] - w0[k]))


def test_prox_needs_an_anchor():
    from bflc_demo_b200.models.mlp import FlatMLP, mlp_spec
    spec = mlp_spec(784, 256, 62)
    t = torch.zeros(spec.total)
    with pytest.raises(ValueError, match="prox_anchor"):
        FlatMLP(spec, t, t.bfloat16(), t.clone(), 128, prox_mu=0.1)
    with pytest.raises(ValueError, match="prox_anchor"):
        FlatMLP(spec, t, t.bfloat16(), t.clone(), 128, prox_mu=0.1, prox_anchor=torch.zeros(3))


def _engine(dtype="fp8", optimizer="adam", sizes=None, alpha=0.0, lr=None, **kw):
    from bflc_demo_b200.data.synthetic import client_sizes, femnist_like
    from bflc_demo_b200.engine.multiclient import MultiClientEngine
    sizes = sizes or client_sizes(20, 1536, sigma=0.8, multiple=256, seed=7)
    cfg = FLConfig(clients=len(sizes), committee_size=4, needed_updates=10, aggregate_count=6, hidden=256,
                   batch_size=256, samples_per_client=max(sizes), val_samples=0, dtype=dtype,
                   optimizer=optimizer, learning_rate=lr or (0.002 if optimizer == "adam" else 0.05),
                   ring_slots=64, non_iid_alpha=alpha, **kw).validate()
    shards = femnist_like(seed=7, noise=48.0, alpha=alpha, sizes=sizes)
    return MultiClientEngine(cfg, shards, device=0)


def _check_weights(eng, blk):
    """Block weights are n_t / sum of the selected n, with n_t = S_t of that client."""
    S = eng.samples_per_client
    sel = blk["selected"]
    total = sum(float(S[t]) for t in sel)
    assert blk["weight"] == [float(np.float32(S[t] / total)) for t in sel], blk


def _standalone(eng, c, g, m, v, base, mu):
    from bflc_demo_b200.models.mlp import FlatMLP
    master = g.clone()
    step = torch.tensor([base], device="cuda", dtype=torch.int32)
    tr = FlatMLP(eng.spec, master, g.to(torch.bfloat16), torch.zeros_like(g), eng.cfg.batch_size,
                 optimizer="adam", lr=eng.cfg.learning_rate, step_dev_ptr=step.data_ptr(), fp8=True,
                 prox_mu=mu, prox_anchor=g if mu > 0 else None)
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
def test_fedprox_clients_in_the_engine():
    """Every client is anchored to the round-start global model: two trained clients (a short and a
    long shard) match a standalone FedProx trainer started from the same state, and differ from
    the same trainer without the term."""
    mu = 0.1
    eng = _engine("fp8", "adam", prox_mu=mu)
    assert eng.server_m is None and eng.server_v is None
    steps = eng.steps_per_client
    done = [0] * eng.cfg.clients
    for rnd in range(2):
        trainers = eng.trainers_now()
        # a one-step client takes its only step at w == anchor, where the term is exactly zero
        multi = [c for c in trainers if steps[c] >= 2]
        picks = [min(multi, key=lambda c: steps[c]), max(multi, key=lambda c: steps[c])]
        assert steps[picks[0]] < steps[picks[1]]
        g = eng.global_master.clone()
        mv = {c: (eng.trainers[c].m.clone(), eng.trainers[c].v.clone()) for c in picks}
        eng.phase_train()
        torch.cuda.synchronize()
        for c in picks:
            master = _standalone(eng, c, g, *mv[c], done[c], mu)
            d = (eng.master[c] - master).abs().max().item()
            assert d < 2e-3 * max(master.abs().max().item(), 1.0), (rnd, c, d)
            assert (eng.master[c] - g).abs().max().item() > 10 * d      # it did train
            plain = _standalone(eng, c, g, *mv[c], done[c], 0.0)
            assert (eng.master[c] - plain).abs().max().item() > 4 * d, (rnd, c, "mu has no effect")
        for c in trainers:
            done[c] += steps[c]
        eng.phase_validate()
        eng.phase_aggregate()
        assert eng.drain_blocks() == []


def _r32(x):
    """Round an fp64 tensor to fp32 and flush subnormals (the kernels build with --use_fast_math)."""
    y = x.float()
    return torch.where(y.abs() < torch.finfo(torch.float32).tiny, torch.zeros_like(y), y).double()


def _f32(x):
    return float(np.float32(x))


def _server_reference(cfg, avg, g, m, v):
    """The server step in fp64 with every fp32 rounding of the kernel's operation order.  Returns
    (g_new, m, v, |update|); g_new is exact for momentum and unrounded for adam / yogi."""
    mode = cfg.server_optimizer
    b1, b2, lr, tau = _f32(cfg.server_beta1), _f32(cfg.server_beta2), _f32(cfg.server_lr), _f32(cfg.server_tau)
    c1, c2 = _f32(1.0 - b1), _f32(1.0 - b2)          # 1 - the fp32 beta, rounded to fp32
    d = _r32(avg - g)
    if mode == "momentum":
        m = _r32(b1 * m + d)
        return _r32(lr * m + g), m, v, None
    m = _r32(b1 * m + _r32(c1 * d))
    d2 = _r32(d * d)
    if mode == "adam":
        v = _r32(b2 * v + _r32(c2 * d2))
    else:
        v = _r32(v - _r32(c2 * d2) * torch.sign(v - d2))
    u = lr * m / (torch.sqrt(v) + tau)
    return g + u, m, v, u.abs()


@gpu
@needs_cuda
@pytest.mark.parametrize("dtype,optimizer,server,server_lr", [
    ("bf16", "sgd", "momentum", 1.0), ("bf16", "sgd", "adam", 0.01), ("bf16", "sgd", "yogi", 0.01),
    ("fp8", "adam", "adam", 0.01)])
def test_server_optimizer_step(dtype, optimizer, server, server_lr):
    """Three rounds phase by phase: the server state m, v matches an fp64 emulation of the fp32
    operation order bit for bit, and so does the momentum step.  Adam / Yogi's step goes through
    the fast-math sqrtf and division: within 0.5 ulp of the new value plus 8 ulp (2^-20) of the
    update's magnitude."""
    eng = _engine(dtype, optimizer, server_optimizer=server, server_lr=server_lr)
    cfg = eng.cfg
    assert eng.server_m is not None and (eng.server_v is not None) == (server != "momentum")
    if eng.server_v is not None:
        assert bool((eng.server_v == _f32(cfg.server_tau * cfg.server_tau)).all())
    for rnd in range(3):
        eng.phase_train()
        eng.phase_validate()
        torch.cuda.synchronize()
        masters = eng.master.clone()
        g = eng.global_master.double()
        m = eng.server_m.double()
        v = eng.server_v.double() if eng.server_v is not None else None
        eng.phase_aggregate()
        torch.cuda.synchronize()
        assert eng.drain_blocks() == []
        blk = eng.host_ledger.blocks()[-1]
        assert blk["selected"], "no client selected: nothing to check"
        avg = torch.zeros(eng.n_params, device="cuda", dtype=torch.float64)
        for t, w in zip(blk["selected"], blk["weight"]):
            avg = (avg + masters[t].double() * _f32(w)).float().double()   # the unchanged FedAvg sum
        g_ref, m_ref, v_ref, u = _server_reference(cfg, avg, g, m, v)
        assert bool((eng.server_m.double() == m_ref).all()), (rnd, "server m")
        if v_ref is not None:
            assert bool((eng.server_v.double() == v_ref).all()), (rnd, "server v")
        got = eng.global_master.double()
        if server == "momentum":
            assert bool((got == g_ref).all()), (rnd, "momentum step")
        else:
            g32 = g_ref.float()
            ulp = (torch.nextafter(g32.abs(), torch.tensor(math.inf, device="cuda")) - g32.abs()).double()
            tol = 0.5 * ulp + u * 2.0 ** -20
            err = (got - g_ref).abs()
            assert bool((err <= tol).all()), (rnd, float((err / tol).max()))
        assert bool((got != avg).any()), "the server step left the average unchanged"
        for c in range(cfg.clients):
            assert torch.equal(eng.master[c], eng.global_master)


# FedAdam's server learning rate for the end-to-end run (20 clients, fp8 + Adam, alpha 0.1, FedProx
# mu 0.01).  On a B200 this run went from 0.02 test accuracy at genesis to 0.55 after 8 rounds; the
# step is about lr per weight per round while |m| / sqrt(v) is near 1.
E2E_SERVER_LR = 0.01


@gpu
@needs_cuda
def test_fedprox_fedadam_end_to_end():
    from bflc_demo_b200.data.synthetic import femnist_like
    from bflc_demo_b200.engine.multiclient import MultiClientEngine
    cfg = FLConfig(clients=20, committee_size=4, needed_updates=10, aggregate_count=6, hidden=256,
                   batch_size=256, samples_per_client=1024, dtype="fp8", optimizer="adam",
                   learning_rate=0.002, ring_slots=64, non_iid_alpha=0.1, prox_mu=0.01,
                   server_optimizer="adam", server_lr=E2E_SERVER_LR).validate()
    eng = MultiClientEngine(cfg, femnist_like(20, 1024, seed=7, noise=48.0, alpha=0.1), device=0)
    test = femnist_like(1, 2048, seed=7, only=0, noise=48.0)[0]
    acc0 = eng.evaluate(test)
    eng.capture()
    for _ in range(8):
        eng.run_round()
    assert eng.drain_blocks() == []
    assert eng.host_ledger.verify_chain() and eng.host_ledger.n_blocks() == 9
    for blk in eng.host_ledger.blocks():
        _check_weights(eng, blk)
    acc = eng.evaluate(test)
    print(f"[fedopt] 20 clients fp8+adam alpha 0.1, FedProx 0.01 + FedAdam lr {E2E_SERVER_LR}: "
          f"acc {acc0:.3f} -> {acc:.3f}")
    assert acc > acc0 + 0.1
