"""CPU tests for the auxiliary subsystems: tracing, metrics, heap layout, data generators."""
import io
import json

import numpy as np
import torch

from bflc_demo_b200.utils.metrics import RunLog
from bflc_demo_b200.utils.tracing import ChromeTrace, PhaseTimer


def test_chrome_trace_and_phase_timer(tmp_path):
    tr = ChromeTrace(rank=3)
    with tr.span("round", epoch=1):
        with tr.span("train"):
            pass
    path = tr.dump(str(tmp_path / "t.json"))
    ev = json.load(open(path))["traceEvents"]
    assert [e["name"] for e in ev] == ["train", "round"] and ev[1]["args"] == {"epoch": 1}
    assert all(e["pid"] == 3 and e["dur"] >= 0 for e in ev)
    t = PhaseTimer()  # without CUDA: a no-op that keeps the API
    with t.phase("x"):
        pass
    s = t.summary()   # (resets the timer: read it once)
    if torch.cuda.is_available():
        assert s["x"]["count"] == 1 and s["x"]["total_ms"] >= 0
    else:
        assert s == {}


def test_runlog_prints_reference_lines(tmp_path):
    buf = io.StringIO()
    log = RunLog(stream=buf, path=str(tmp_path / "m.jsonl"))
    log.round(9, 5.96238, test_acc=0.9214)
    out = buf.getvalue()
    assert "the 9 epoch , global loss : 5.962380" in out      # CommitteePrecompiled.cpp:424
    assert "Epoch: 009, test_acc: 0.9214" in out              # python-sdk/main.py:327
    log.close()
    row = json.loads(open(tmp_path / "m.jsonl").read())
    assert row["epoch"] == 9 and abs(row["test_acc"] - 0.9214) < 1e-9


def test_heap_layout_is_aligned_and_disjoint():
    from bflc_demo_b200.parallel.layout import HeapLayout
    lay = HeapLayout(217_216, ring_slots=64)
    offs = sorted(lay.offsets.items(), key=lambda kv: kv[1])
    for (name, off), (_, nxt) in zip(offs, offs[1:]):
        assert off % 16 == 0 and off < nxt, name
    for k in ("work_master", "work_shadow", "upload_master0", "upload_shadow1", "global"):
        assert lay.offsets[k] % 4096 == 0
    assert lay.total_bytes % (2 << 20) == 0
    fd = lay.fed_dict(1, 4, [10, 20, 30, 40], 0)
    assert fd["upload_master_off"] == [lay.offsets["upload_master0"], lay.offsets["upload_master1"]]
    assert fd["n_params"] == 217_216


def test_synthetic_generators_shapes_and_skew():
    from bflc_demo_b200.data.synthetic import cifar_like, femnist_like, occupancy_like, tokens_like
    sh = femnist_like(4, 64, seed=1)
    assert len(sh) == 4 and sh[0].x.shape == (64, 784) and sh[0].x.dtype == torch.uint8
    assert int(sh[0].y.max()) < 62
    non_iid = cifar_like(4, 400, seed=1, alpha=0.1)
    iid = cifar_like(4, 400, seed=1, alpha=0.0)
    assert non_iid[0].x.shape == (400, 3, 32, 32)
    h_non = np.bincount(non_iid[0].y.numpy(), minlength=10) / 400
    h_iid = np.bincount(iid[0].y.numpy(), minlength=10) / 400
    assert h_non.max() > h_iid.max() + 0.1         # Dirichlet(0.1) label skew
    tk = tokens_like(2, 16, seq_len=128)
    assert tk[0].x.shape == (16, 128) and int(tk[0].x.max()) < 30522
    x, y = occupancy_like()
    assert x.shape == (8143, 5) and 0.15 < y.mean() < 0.28


def test_param_spec_offsets_are_tma_aligned():
    from bflc_demo_b200.models.mlp import mlp_spec
    from bflc_demo_b200.models.nets import BertBase, LeNet5, ResNet18
    for spec in (mlp_spec(784, 256, 62), LeNet5(10).spec, ResNet18(10).spec, BertBase(2, layers=1).spec):
        assert spec.total % 8 == 0
        for e in spec.entries:
            assert e.offset % 8 == 0
            if len(e.shape) == 2:
                assert e.shape[1] % 8 == 0, e.name   # row pitch = 16-byte multiple in bf16
    flat = torch.empty(mlp_spec().total)
    mlp_spec().init_(flat, seed=3)
    flat2 = torch.empty(mlp_spec().total)
    mlp_spec().init_(flat2, seed=3)
    assert torch.equal(flat, flat2)                  # identical genesis on every rank


def test_implicit_conv_eligibility_and_pixel_tiles():
    """Host-side geometry of the implicit-GEMM convolution (ops/nn.py mirrors
    csrc/kernels/gemm_sm100.cu::conv_pixel_tile): a pixel tile is whole image rows."""
    from bflc_demo_b200.ops import nn as F
    assert F._pix_tile(128, 32, 32) and F._pix_tile(64, 32, 32)      # 4 / 2 rows of one image
    assert F._pix_tile(128, 16, 16) and F._pix_tile(128, 8, 8)       # 8 rows; two whole 8x8 images
    assert F._pix_tile(128, 4, 4) and F._pix_tile(64, 4, 4)          # 8 / 4 whole 4x4 images
    assert not F._pix_tile(128, 28, 28)                              # 128 % 28 != 0
    assert not F._pix_tile(128, 12, 16)                              # 8 rows do not divide 12
    assert not F._pix_tile(64, 7, 128)                               # a row is wider than the tile
    # ResNet-18 body layers are eligible; the stem (Cin = 3) and LeNet (Cin = 3 / 6, 5x5) are not
    assert F.conv_is_implicit(32, 32, 64, 3, 3, 1, 1, 9 * 64)
    assert F.conv_is_implicit(32, 32, 64, 3, 3, 2, 1, 9 * 64)
    assert F.conv_is_implicit(16, 16, 128, 1, 1, 2, 0, 128)
    assert not F.conv_is_implicit(32, 32, 3, 3, 3, 1, 1, 32)
    assert not F.conv_is_implicit(14, 14, 6, 5, 5, 1, 0, 152)
    prev = F.set_precision("mx8")                                    # fp8 forward keeps the im2col path
    try:
        assert not F.conv_is_implicit(32, 32, 64, 3, 3, 1, 1, 9 * 64)
    finally:
        F.set_precision(prev)


def test_round_state_mirror_layout_matches_the_native_struct():
    """run_round_e2e parses the pinned mirror page with one precompiled struct."""
    from bflc_demo_b200._native import C
    from bflc_demo_b200.engine.fused import _ROUND_STATE
    sz = C().struct_sizes()
    assert _ROUND_STATE.size == sz["RoundState"]
    assert sz["state_epoch_off"] == 0 and sz["state_role_off"] == 16
    assert sz["state_global_loss_off"] == 84 and sz["state_digest_off"] == 88
    assert sz["kMirrorSeqWord"] * 4 >= sz["RoundState"]


def test_vector_ranges_cover_exactly_the_1d_parameters():
    """The committee pulls the bf16 copy of a candidate plus only these fp32 ranges
    (engine/generic.py::vector_ranges -> fed_pull_candidates)."""
    from bflc_demo_b200.engine.generic import vector_ranges
    from bflc_demo_b200.models.nets import build_model
    for name, kw in (("lenet5", {}), ("resnet18", {}), ("bert", {"layers": 2})):
        spec = build_model(name, 10, **kw).spec
        r = vector_ranges(spec)
        assert r.dtype == torch.int64 and r.shape[1] == 2 and (r[:, 1] > 0).all()
        lo, hi = r[:, 0] * 4, (r[:, 0] + r[:, 1]) * 4
        assert (lo[1:] > hi[:-1]).all()                      # sorted, coalesced, disjoint
        covered = torch.zeros(spec.total + 8, dtype=torch.bool)
        for a, b in zip(lo.tolist(), hi.tolist()):
            assert b <= spec.total + 3
            covered[a:b] = True
        for e in spec.entries:
            seg = covered[e.offset:e.offset + e.numel]
            if len(e.shape) == 1:
                assert seg.all(), e.name                     # every 1-D parameter is pulled in fp32
            else:
                # a matrix is never pulled in fp32, except for the <= 3 elements a rounded-up
                # neighbouring range may touch at its very start (alignment padding makes that 0)
                assert int(seg.sum()) == 0, e.name
        frac = float((hi - lo).sum()) / spec.total
        assert frac < 0.02 if name != "lenet5" else frac < 0.1
