"""C++ ledger runtime vs the pure-Python oracle (SURVEY.md 4: the reference has no tests;
the protocol of section 1.3 is the spec, every guard path is exercised here)."""
import itertools

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from bflc_demo_b200._native import ledger as _ledger
from bflc_demo_b200.protocol import oracle as O

L = _ledger()


def make(client_num=8, comm=3, agg=4, needed=5, model_size=12, lr=0.001, wbs=0, solo=0, seed=0):
    c = L.LedgerConfig()
    c.client_num, c.comm_count, c.aggregate_count, c.needed_update_count = client_num, comm, agg, needed
    c.model_size, c.learning_rate, c.weight_by_score, c.solo, c.seed = model_size, lr, wbs, solo, seed
    led = L.Ledger(c)
    orc = O.OracleLedger(client_num, comm, agg, needed, lr, model_size, bool(wbs), bool(solo))
    return led, orc


def S(x):
    return int(x)


def test_config_validation():
    c = L.LedgerConfig()
    assert c.validate() == ""  # the reference constants 20/4/6/10 are valid
    c.needed_update_count = 17
    assert "needed_update_count" in c.validate()
    c.needed_update_count = 10
    c.aggregate_count = 11
    assert c.validate() != ""
    with pytest.raises(ValueError):
        L.Ledger(c)


def test_genesis_and_registration():
    led, orc = make()
    assert led.epoch() == L.EPOCH_NOT_STARTED == -999  # C:322
    model, ep = led.QueryGlobalModel()
    assert ep == -999 and np.all(model == 0) and model.size == 12  # zero model, C:325-327
    # unknown caller is reported as trainer and not persisted (C:197-200)
    assert led.QueryState(5) == (L.ROLE_TRAINER, -999)
    # uploads before start are dropped
    assert led.UploadLocalUpdate(0, np.zeros(12, np.float32), 1, 0.0, -999) == L.Status.NOT_STARTED
    for i in range(8):
        assert led.RegisterNode(i) == L.Status.OK
        assert orc.RegisterNode(i) == O.OK
        assert led.epoch() == (0 if i == 7 else -999)
    assert led.RegisterNode(3) == L.Status.OK  # idempotent, C:171
    assert led.RegisterNode(99) == L.Status.UNKNOWN_CLIENT
    roles = led.roles()
    assert roles == [orc.role[i] for i in range(8)]
    assert sum(r == L.ROLE_COMM for r in roles) == 3


def run_round(led, orc, rng, model_size=12, byz=None):
    ep = led.epoch()
    roles = led.roles()
    trainers = [i for i, r in enumerate(roles) if r & L.ROLE_TRAINER]
    comm = [i for i, r in enumerate(roles) if r & L.ROLE_COMM]
    for t in trainers:
        d = rng.standard_normal(model_size).astype(np.float32)
        n, c = int(rng.integers(50, 400)), float(rng.random())
        s1 = led.UploadLocalUpdate(t, d, n, c, ep)
        s2 = orc.UploadLocalUpdate(t, d, n, c, ep)
        assert S(s1) == s2
    ups = led.QueryAllUpdates()
    assert [u["sender"] for u in ups] == [u["sender"] for u in orc.QueryAllUpdates()]
    admitted = [u["sender"] for u in ups]
    last = None
    for c in comm:
        row = {t: float(np.float32(rng.random())) for t in admitted}
        s1 = led.UploadScores(c, ep, row)
        s2 = orc.UploadScores(c, ep, row)
        assert S(s1) == s2
        last = s1
    assert last == L.Status.AGGREGATED
    return admitted


@pytest.mark.parametrize("cfg", [dict(), dict(client_num=4, comm=2, agg=2, needed=2),
                                 dict(client_num=20, comm=4, agg=6, needed=10),
                                 dict(client_num=2, comm=1, agg=1, needed=1),
                                 dict(client_num=1, comm=1, agg=1, needed=1, solo=1),
                                 dict(wbs=1)])
def test_rounds_match_oracle(cfg):
    led, orc = make(**cfg)
    n = cfg.get("client_num", 8)
    for i in range(n):
        led.RegisterNode(i); orc.RegisterNode(i)
    rng = np.random.default_rng(1)
    for rnd in range(6):
        run_round(led, orc, rng)
        assert led.epoch() == orc.epoch == rnd + 1
        assert led.roles() == [orc.role[i] for i in range(n)]
        m, _ = led.QueryGlobalModel()
        np.testing.assert_allclose(m, orc.global_model, rtol=1e-5, atol=1e-7)
        blk = led.blocks()[-1]
        h = orc.history[-1]
        assert blk["selected"] == h["selected"]
        np.testing.assert_allclose(blk["weight"], [h["weight"][t] for t in h["selected"]], rtol=1e-6)
        assert abs(blk["global_loss"] - h["global_loss"]) < 1e-6
        assert led.update_count() == 0 and led.score_count() == 0  # reset, C:427-441
    assert led.verify_chain()
    assert led.n_blocks() == 6


def test_guards():
    led, orc = make()
    for i in range(8):
        led.RegisterNode(i)
    roles = led.roles()
    trainers = [i for i, r in enumerate(roles) if r == L.ROLE_TRAINER]
    comm = [i for i, r in enumerate(roles) if r == L.ROLE_COMM]
    z = np.zeros(12, np.float32)
    assert led.UploadLocalUpdate(trainers[0], z, 1, 0.0, 1) == L.Status.STALE_EPOCH        # C:225
    assert led.UploadLocalUpdate(trainers[0], z[:5], 1, 0.0, 0) == L.Status.BAD_PAYLOAD
    assert led.UploadLocalUpdate(comm[0], z, 1, 0.0, 0) == L.Status.NOT_TRAINER
    assert led.UploadLocalUpdate(trainers[0], z, 1, 0.0, 0) == L.Status.OK
    assert led.UploadLocalUpdate(trainers[0], z, 1, 0.0, 0) == L.Status.DUPLICATE          # C:232
    assert led.QueryAllUpdates() == []                                                     # C:304-307
    assert led.UploadScores(comm[0], 0, {trainers[0]: 0.5}) == L.Status.NOT_READY
    for t in trainers[1:]:
        assert led.UploadLocalUpdate(t, z, 1, 0.0, 0) == L.Status.OK
    assert len(led.QueryAllUpdates()) == 5
    assert led.UploadScores(trainers[0], 0, {}) == L.Status.NOT_COMMITTEE                  # C:274
    assert led.UploadScores(comm[0], 3, {}) == L.Status.STALE_EPOCH                        # C:268
    row = {t: 0.5 for t in trainers}
    assert led.UploadScores(comm[0], 0, row) == L.Status.OK
    # duplicate row: replaces, does NOT advance the count (reference bug C:279-289 not emulated)
    assert led.UploadScores(comm[0], 0, row) == L.Status.OK
    assert led.score_count() == 1
    assert led.UploadScores(comm[1], 0, {trainers[0]: float("nan")}) == L.Status.BAD_PAYLOAD
    assert led.UploadScores(comm[1], 0, row) == L.Status.OK
    assert led.UploadScores(comm[2], 0, row) == L.Status.AGGREGATED
    assert led.epoch() == 1
    c = led.counters()
    assert c["aggregations"] == 1 and c["uploads_rejected"] == 4 and c["uploads_ok"] == 5
    log = led.drain_log()
    assert any("global loss" in s for s in log) and any("not collected" in s for s in log)


def test_first_k_admission_quota():
    # 20 clients, 16 trainers, only the first 10 uploads are admitted (C:239)
    led, orc = make(client_num=20, comm=4, agg=6, needed=10)
    for i in range(20):
        led.RegisterNode(i)
    trainers = [i for i, r in enumerate(led.roles()) if r == L.ROLE_TRAINER]
    z = np.zeros(12, np.float32)
    st_ = [led.UploadLocalUpdate(t, z, 1, 0.0, 0) for t in reversed(trainers)]
    assert st_[:10] == [L.Status.OK] * 10 and st_[10:] == [L.Status.QUOTA_FULL] * 6
    assert [u["sender"] for u in led.QueryAllUpdates()] == list(reversed(trainers))[:10]


def test_true_median_is_order_independent():
    """Spec deviation (SURVEY.md 1.3): the reference's quickselect `GetMid` (C:81-115) tests
    parity on a mutated bound and is input-order dependent (e.g. {5,1,9} -> 7, lower median for
    some orderings of 4 values).  It is NOT emulated anywhere in this repo; every implementation
    (oracle, C++ ledger / device math via run_consensus) returns the true median for every
    ordering, even and odd counts."""
    assert O.true_median([5, 1, 9]) == 5
    for vals, want in (([1.0, 2.0, 3.0, 4.0], 2.5), ([5.0, 1.0, 9.0], 5.0), ([0.25, 0.75], 0.5)):
        n = len(vals)
        for p in itertools.permutations(vals):
            assert O.true_median(list(p)) == want
            # committee ranks 0..n-1 score the single trainer n with the permuted values
            role = [L.ROLE_COMM] * n + [L.ROLE_TRAINER]
            rows = [[0.0] * (n + 1) for _ in range(n + 1)]
            scored = [[0] * (n + 1) for _ in range(n + 1)]
            for c in range(n):
                rows[c][n] = p[c]
                scored[c][n] = 1
            out = L.run_consensus(n + 1, n, 1, False, role, [0] * n + [1], rows, scored,
                                  [1] * (n + 1), [0.0] * (n + 1))
            assert out["median"][n] == want


def test_snapshot_restore_and_replica_hash():
    led, orc = make()
    led2, _ = make()
    for i in range(8):
        led.RegisterNode(i); orc.RegisterNode(i); led2.RegisterNode(i)
    rng = np.random.default_rng(7)
    run_round(led, orc, rng)
    blob = led.snapshot()
    back = L.Ledger.restore(blob)
    assert back.state_hash() == led.state_hash() and back.epoch() == 1 and back.verify_chain()
    # corrupt one byte of the last block -> restore must refuse
    bad = bytearray(blob); bad[-40] ^= 1
    with pytest.raises(RuntimeError):
        L.Ledger.restore(bytes(bad))
    # two replicas fed the same transactions in the same order agree bit-for-bit
    rng = np.random.default_rng(7)
    _, orc2 = make()
    for i in range(8):
        orc2.RegisterNode(i)
    run_round(led2, orc2, rng)
    assert led2.state_hash() == led.state_hash()
    assert led2.blocks()[-1]["hash"] == led.blocks()[-1]["hash"]


def test_sha256_vectors():
    assert L.sha256_hex(b"") == "e3b0c44298fc1c149afbf4c8996fb92427ae41e4649b934ca495991b7852b855"
    assert L.sha256_hex(b"abc") == "ba7816bf8f01cfea414140de5dae2223b00361a396177a9cb410ff61f20015ad"
    import hashlib
    for n in (55, 56, 63, 64, 65, 1000):
        b = bytes(range(256)) * 4
        assert L.sha256_hex(b[:n]) == hashlib.sha256(b[:n]).hexdigest()


@settings(max_examples=200, deadline=None)
@given(st.data())
def test_consensus_math_matches_oracle(data):
    n = data.draw(st.integers(1, 10))
    n_comm = data.draw(st.integers(1, n))
    role = {}
    comm_set = set(data.draw(st.permutations(range(n)))[:n_comm])
    for r in range(n):
        role[r] = O.ROLE_COMM if r in comm_set else O.ROLE_TRAINER
    trainers = [r for r in range(n) if role[r] == O.ROLE_TRAINER]
    admitted = [t for t in trainers if data.draw(st.booleans())] if trainers else []
    n_agg = data.draw(st.integers(1, max(1, n)))
    grid = st.sampled_from([0.0, 0.25, 0.5, 0.5, 0.75, 1.0])  # force ties
    scores = {c: {t: data.draw(grid) for t in admitted if data.draw(st.integers(0, 9)) > 0} for c in comm_set}
    ns = {t: data.draw(st.integers(0, 500)) for t in admitted}
    ac = {t: data.draw(st.floats(0, 10, width=32)) for t in admitted}
    wbs = data.draw(st.booleans())
    ref = O.run_consensus(n, n_comm, n_agg, role, admitted, scores, ns, ac, wbs)
    score_m = [[scores.get(c, {}).get(t, 0.0) for t in range(n)] for c in range(n)]
    scored_m = [[1 if t in scores.get(c, {}) else 0 for t in range(n)] for c in range(n)]
    got = L.run_consensus(n, n_comm, n_agg, wbs, [role[r] for r in range(n)],
                          [1 if r in admitted else 0 for r in range(n)], score_m, scored_m,
                          [ns.get(r, 0) for r in range(n)], [ac.get(r, 0.0) for r in range(n)])
    assert got["order"] == ref.order
    assert got["selected"] == ref.selected
    assert got["role_after"] == [ref.role_after[r] for r in range(n)]
    for t in admitted:
        assert abs(got["median"][t] - ref.median[t]) < 1e-6
    for t in ref.selected:
        assert abs(got["weight"][t] - ref.weight[t]) < 1e-6
    assert abs(got["global_loss"] - ref.global_loss) < 1e-4


def test_device_round_and_snapshot_inputs_are_validated():
    """Untrusted inputs of the host ledger: a short device record is refused (no out-of-bounds
    read), and a corrupted snapshot either restores or raises -- it never names a client id
    outside [0, client_num) (those ids index fixed arrays in the aggregation)."""
    led, orc = make()
    for i in range(8):
        led.RegisterNode(i); orc.RegisterNode(i)
    roles = led.roles()
    rec = dict(epoch=0, role_before=roles, role_after=roles, score_rows=[[0.0] * 8] * 8, scored_mask=[0] * 8,
               n_samples=[1] * 8, avg_cost=[0.0] * 8, admitted_mask=0, selected_mask=0, global_loss=0.0,
               model_digest=0, weight_by_score=0)
    for key, short in (("n_samples", [1] * 3), ("avg_cost", [0.0]), ("scored_mask", []),
                       ("score_rows", [[0.0] * 8] * 7 + [[0.0] * 2]), ("role_after", roles[:4])):
        bad = dict(rec); bad[key] = short
        assert "short" in led.AppendDeviceRound(bad), key
    assert led.epoch() == 0                      # nothing was appended
    rng = np.random.default_rng(3)
    run_round(led, orc, rng)
    blob = bytes(led.snapshot())
    assert L.Ledger.restore(blob).state_hash() == led.state_hash()
    ok = bad_n = 0
    for _ in range(300):
        b = bytearray(blob)
        for _ in range(int(rng.integers(1, 4))):
            b[int(rng.integers(8, len(b)))] = int(rng.integers(0, 256))
        try:
            r = L.Ledger.restore(bytes(b))
            assert all(0 <= c < 8 for c in range(len(r.roles())))
            ok += 1
        except (RuntimeError, ValueError, MemoryError):
            bad_n += 1
    assert ok + bad_n == 300 and bad_n > 0
    with pytest.raises(RuntimeError):
        L.Ledger.restore(blob[: len(blob) // 2])
    # a model size the blob cannot hold (int64 at byte 28) is refused before the model is allocated
    huge = bytearray(blob)
    huge[28:36] = (1 << 40).to_bytes(8, "little")
    with pytest.raises(RuntimeError, match="model size"):
        L.Ledger.restore(bytes(huge))
