"""2-layer MLP 784 -> hidden -> 62 (BASELINE.json configs #1/#2), hand-scheduled: every
forward/backward GEMM is the tcgen05 kernel with a fused epilogue, the whole training step
is six launches and is CUDA-graph capturable (no host syncs, no allocations).

Reference parity: the reference's model is the degenerate single-layer case
``pred = x @ W + b`` with softmax-cross-entropy and plain SGD, batch 100, one pass per
round (python-sdk/main.py:109-148); ``SoftmaxRegression`` below is exactly that model.

  step(x, y):
    1. h       = relu(x @ W1^T + b1)                    GEMM  (bias+ReLU epilogue)
    2. dlogits = softmax(h @ W2^T + b2) - onehot(y)     GEMM  (xent epilogue: loss, #correct,
                                                              db2 column sums)
    3. dW2     = dlogits^T @ h                          GEMM  (MN-major A and B, split-K)
    4. dh      = (dlogits @ W2) * (h > 0)               GEMM  (MN-major B, ReLU-bwd mask, db1)
    5. dW1     = dh^T @ x                               GEMM  (MN-major A and B, split-K)
    6. SGD / Adam over the flat buffer (+ bf16 shadow refresh + grad zeroing)
"""
from __future__ import annotations

from typing import Optional

import torch

from .._native import C
from ..ops import gemm as G
from .flat import ParamSpec


def sf_bytes(rows: int, K: int) -> int:
    """Bytes of the MXFP8 scale-chunk array of a [rows, K] operand: one 512-byte chunk per
    (128 rows, 128 K) -- csrc/include/epi_common.cuh."""
    return -(-rows // 128) * -(-K // 128) * 512


def mlp_spec(in_dim: int = 784, hidden: int = 256, n_classes: int = 62) -> ParamSpec:
    return ParamSpec([("w1", (hidden, in_dim)), ("b1", (hidden,)),
                      ("w2", (n_classes, hidden)), ("b2", (n_classes,))])


def softmax_regression_spec(n_features: int = 5, n_class: int = 2) -> ParamSpec:
    """The reference model: W[n_features, n_class] stored [out, in] + b (H:7-8, M:113-120)."""
    return ParamSpec([("w", (n_class, n_features)), ("b", (n_class,))])


class FlatMLP:
    """Fused-kernel trainer over flat buffers.  ``master``/``shadow``/``grad`` are 1-D tensors
    of ``spec.total`` elements (fp32 / bf16 / fp32); they may live in the symmetric heap.

    ``prox_mu`` > 0 (FedProx): every step adds ``prox_mu * (w - prox_anchor)`` to the gradient, the
    gradient of ``prox_mu / 2 * ||w - prox_anchor||^2``.  ``prox_anchor`` is an fp32 tensor with the
    master's layout (the global model at round start) that stays fixed while the trainer runs.  The
    reported loss stays the cross-entropy alone."""

    def __init__(self, spec: ParamSpec, master: torch.Tensor, shadow: torch.Tensor,
                 grad: torch.Tensor, batch: int, *, optimizer: str = "sgd", lr: float = 1e-3,
                 loss_sum: Optional[torch.Tensor] = None, correct: Optional[torch.Tensor] = None,
                 step_dev_ptr: int = 0, fp8: bool = False, prox_mu: float = 0.0,
                 prox_anchor: Optional[torch.Tensor] = None):
        if prox_mu < 0 or (prox_mu > 0 and prox_anchor is None):
            raise ValueError("prox_mu must be >= 0, and prox_mu > 0 needs a prox_anchor")
        if prox_anchor is not None and (prox_anchor.shape != master.shape or prox_anchor.dtype != torch.float32):
            raise ValueError("prox_anchor: fp32 with the master's shape")
        self.prox_mu = float(prox_mu)
        self.prox_anchor = prox_anchor if self.prox_mu > 0 else None
        self.spec, self.master, self.shadow, self.grad = spec, master, shadow, grad
        self.p = spec.views(master)
        self.s = spec.views(shadow)
        self.g = spec.views(grad)
        self.hidden, self.in_dim = spec.by_name["w1"].shape
        self.n_classes = spec.by_name["w2"].shape[0]
        self.batch = batch
        dev = master.device
        self.h = torch.empty(batch, self.hidden, device=dev, dtype=torch.bfloat16)
        self.dh = torch.empty(batch, self.hidden, device=dev, dtype=torch.bfloat16)
        self.ncp = (self.n_classes + 7) // 8 * 8          # dlogits row stride (TMA alignment)
        self.dlogits = torch.zeros(batch, self.ncp, device=dev, dtype=torch.bfloat16)
        self.loss_sum = loss_sum if loss_sum is not None else torch.zeros(1, device=dev)
        self.correct = correct if correct is not None else torch.zeros(1, device=dev, dtype=torch.int32)
        self.optimizer, self.lr = optimizer, lr
        self.m = torch.zeros_like(master) if optimizer == "adam" else None
        self.v = torch.zeros_like(master) if optimizer == "adam" else None
        self.step_dev_ptr = step_dev_ptr
        # weight-gradient GEMMs reduce over the batch: split the reduction only when it is long
        # (measured on B200: at batch 512 the unsplit 64-wide-tile launch is faster, see profiles/)
        k_blocks = (batch + 63) // 64
        self.split_k = 1 if k_blocks <= 16 else max(1, min(8, k_blocks // 8))
        self.side = torch.cuda.Stream(device=dev)
        self._ev_fork = torch.cuda.Event()
        self._ev_join = torch.cuda.Event()
        # block-scaled fp8 forward (persistent trainer only): this trainer's quantised weights
        # (an Mx8MlpLayout blob, refreshed by the optimizer epilogue) and the per-step e4m3 h
        self.fp8 = bool(fp8)
        self.ql = C().mx8_mlp_layout(self.in_dim, self.hidden) if self.fp8 else None
        if self.fp8:
            self.work_q = torch.zeros(self.ql["total"], device=dev, dtype=torch.uint8)
            self.h_q = torch.zeros(batch, self.hidden, device=dev, dtype=torch.uint8)
            self.h_sf = torch.full((sf_bytes(batch, self.hidden),), 127, device=dev, dtype=torch.uint8)

    # -------------------------------------------------------------- training
    def forward_backward(self, x: torch.Tensor, y: torch.Tensor) -> None:
        """x: bf16 [batch, in_dim], y: int32 [batch].  Accumulates grads into ``grad``."""
        B = x.shape[0]
        s, g = self.s, self.g
        h = self.h[:B]
        G.gemm(x, s["w1"], out=h, bias=self.p["b1"], act=G.ACT_RELU)
        dl = self.dlogits[:B]
        G.gemm_xent(h, s["w2"], y, n_classes=self.n_classes, bias=self.p["b2"], dlogits=dl,
                    grad_scale=1.0 / B, loss_sum=self.loss_sum, correct=self.correct,
                    colsum=g["b2"])
        # dW2 and dh are independent (both only read dlogits, h, W2): dW2 runs on a side stream
        # (a parallel branch of the captured graph) while dh -> dW1 stay on the main stream.
        main = torch.cuda.current_stream()
        self._ev_fork.record(main)
        self.side.wait_event(self._ev_fork)
        with torch.cuda.stream(self.side):
            # dW2[c, j] = sum_b dlogits[b, c] h[b, j]
            G.gemm(dl[:, :self.n_classes], h, out=g["w2"], a_mn=True, b_mn=True,
                   split_k=self.split_k)
            self._ev_join.record(self.side)
        # dh = (dlogits @ W2) * relu'(h);  db1 = colsum(dh)
        G.gemm(dl[:, :self.n_classes], s["w2"], out=self.dh[:B], b_mn=True, aux_in=h, act_bwd=1,
               colsum=g["b1"])
        # dW1 = dh^T @ x
        G.gemm(self.dh[:B], x, out=g["w1"], a_mn=True, b_mn=True, split_k=self.split_k)
        main.wait_event(self._ev_join)

    def optimizer_step(self, step_in_round: int = 1) -> None:
        C().optim_step(self.optimizer == "adam", self.master, self.grad, self.shadow, self.m,
                       self.v, self.lr, 0.0, 0.9, 0.999, 1e-8, step_in_round, self.step_dev_ptr, 0,
                       True)

    def train_epoch(self, X: torch.Tensor, Y: torch.Tensor, steps: int) -> None:
        """One pass: ``steps`` mini-batches of ``batch`` rows, remainder dropped (M:141-148)."""
        B = self.batch
        for i in range(steps):
            self.forward_backward(X[i * B:(i + 1) * B], Y[i * B:(i + 1) * B])
            if self.prox_mu > 0:
                self.grad.add_(self.master - self.prox_anchor, alpha=self.prox_mu)
            self.optimizer_step(i + 1)

    def fused_ok(self, steps: int) -> bool:
        """Shape limits of the persistent one-launch trainer (csrc/kernels/mlp_round_sm100.cu)."""
        B, H, D = self.batch, self.hidden, self.in_dim
        mt_b, nt_h, nt_d, mt_h = -(-B // 128), -(-H // 64), -(-D // 64), -(-H // 128)
        need = max(mt_b * nt_h, mt_h * nt_d + nt_h + 1)
        return (need <= 128 and B % 8 == 0 and H % 8 == 0 and D % 8 == 0 and self.n_classes <= 64)

    def offsets(self):
        e = self.spec.by_name
        return [e["w1"].offset, e["b1"].offset, e["w2"].offset, e["b2"].offset]

    def quantize_weights(self, master: Optional[torch.Tensor] = None,
                         blob: Optional[torch.Tensor] = None) -> torch.Tensor:
        """fp32 master weights -> MXFP8 blob (e4m3 + UE8M0 scale chunks + fp32 biases).  Run at
        the start of every round: the consensus kernel has just rewritten the training buffers."""
        blob = self.work_q if blob is None else blob
        C().quantize_mlp_blob(self.master if master is None else master, self.offsets(), self.in_dim,
                              self.hidden, self.n_classes, blob)
        return blob

    def train_epoch_fused(self, X: torch.Tensor, Y: torch.Tensor, steps: int,
                          barrier_ptr: int, dbg: Optional[torch.Tensor] = None, plan: int = -1,
                          epiopt: int = -1, x_ready_ptr: int = 0, round_seq_ptr: int = 0,
                          x_q: Optional[torch.Tensor] = None, x_sf: Optional[torch.Tensor] = None,
                          fed: Optional[dict] = None, upq_off=(), n_samples: int = 0,
                          n_loss_terms: int = 0, byz_mode: int = 0, byz_scale: float = 0.0,
                          straggle_us: int = 0) -> None:
        """All ``steps`` mini-batch steps in ONE persistent kernel launch; ``barrier_ptr`` is a
        device uint32 that is zero on entry (the phase barrier).  ``dbg``: optional int64
        [steps, 32] buffer that receives %globaltimer phase stamps of CTA 0.  ``plan`` /
        ``epiopt`` pick a phase plan explicitly (0 | 1 | 3 | 4, 0 | 1; -1 = BFLC_MLP_CHAIN /
        BFLC_MLP_EPIOPT / default) -- all plans are numerically equivalent.  ``x_ready_ptr`` /
        ``round_seq_ptr`` (device uint32[steps] / uint32): the producer of step s waits until
        ``x_ready[s] >= *round_seq`` (input pipeline, engine/fused.py).

        ``x_q`` / ``x_sf`` (fp8 trainers): the e4m3 copy of X and its scale chunks
        (``prep_inputs``); fwd1 / fwd2 then run block-scaled fp8.  ``fed`` (+ ``upq_off``,
        ``n_samples``, ...): fuse UploadLocalUpdate into the last step (the optimizer epilogue
        writes the upload buffers, CTA 0 releases FLAG_TRAINED on every peer)."""
        C().mlp_round(X, Y, self.master, self.shadow, self.grad, self.offsets(), self.h, self.dlogits,
                      self.dh, self.loss_sum, self.correct, barrier_ptr, self.batch, steps,
                      self.in_dim, self.hidden, self.n_classes, self.lr,
                      self.optimizer == "adam", self.m, self.v, self.step_dev_ptr, dbg, plan, epiopt,
                      x_ready_ptr, round_seq_ptr,
                      x_q if self.fp8 else None, x_sf if self.fp8 else None,
                      self.work_q if self.fp8 else None, self.h_q if self.fp8 else None,
                      self.h_sf if self.fp8 else None, fed, list(upq_off), n_samples, n_loss_terms,
                      byz_mode, byz_scale, straggle_us, prox_mu=self.prox_mu,
                      prox_anchor=self.prox_anchor)

    # ------------------------------------------------------------ evaluation
    def accuracy_counts(self, X: torch.Tensor, Y: torch.Tensor, shadow: Optional[torch.Tensor] = None,
                        master: Optional[torch.Tensor] = None) -> torch.Tensor:
        """#correct of (optionally another model's) weights on (X, Y) -> int32 [1] (K6)."""
        s = self.spec.views(shadow) if shadow is not None else self.s
        p = self.spec.views(master) if master is not None else self.p
        n = X.shape[0]
        h = torch.empty(n, self.hidden, device=X.device, dtype=torch.bfloat16)
        G.gemm(X, s["w1"], out=h, bias=p["b1"], act=G.ACT_RELU)
        cnt = torch.zeros(1, device=X.device, dtype=torch.int32)
        G.gemm_argmax_acc(h, s["w2"], Y, cnt, n_classes=self.n_classes, bias=p["b2"])
        return cnt


def torch_reference_step(params: dict, x: torch.Tensor, y: torch.Tensor, lr: float):
    """Plain fp32 PyTorch version of one SGD step of the same MLP (numerics oracle)."""
    w1, b1, w2, b2 = (params[k].detach().clone().requires_grad_(True) for k in ("w1", "b1", "w2", "b2"))
    h = torch.relu(x.float() @ w1.t() + b1)
    logits = h @ w2.t() + b2
    loss = torch.nn.functional.cross_entropy(logits, y.long())
    loss.backward()
    new = {k: (t - lr * t.grad).detach() for k, t in (("w1", w1), ("b1", b1), ("w2", w2), ("b2", b2))}
    grads = {"w1": w1.grad, "b1": b1.grad, "w2": w2.grad, "b2": b2.grad}
    return loss.detach(), new, grads
