"""One whole training iteration as a single replayable unit: forward (batch-statistics BatchNorm, dropout), the fused
losses, the full backward, the bucketed gradient all-reduce and the optimiser step.

Replaces the body of the reference's training loop, ``/root/reference/src/train.py:94-141`` (single process) and
``/root/reference/src/multi_gpu_train2.py:139-196`` (one rank of the data-parallel job):

    outs = model(imgs); ...eight losses...; optimizer.zero_grad(); loss.backward(); optimizer.step()

The step is enqueued without any host synchronisation and -- by default -- captured once into a CUDA graph, so that the
~1000 kernel launches of an iteration cost one ``cudaGraphLaunch`` on the host. ``model(x)`` + ``HeatmapLoss`` +
``loss.backward()`` (autograd) remain available and produce the same numbers; this class is the fast path.
"""
from __future__ import annotations

import os
from typing import Sequence

import torch

from . import _lib
from .loss import ATOM_TYPE_WEIGHTS, loss_forward_backward, loss_forward_p8, p8_loss_supported


class TrainStep:
    """step = TrainStep(model, optimizer, class_weights=True, buckets=None, use_graph=True)
    loss = step(imgs, targets)        # imgs [B,1,H,W] fp32/uint8 CUDA, targets = the 8 dense maps of utils.collate_fn

    ``optimizer`` may be None (gradients are left in ``p.grad``). With ``use_graph`` the optimiser must be constructed
    with ``capturable=True`` to be part of the graph; otherwise it is stepped eagerly after the replay.
    ``buckets`` is an ``abcnet_b200.ddp.GradBuckets`` over ``model.parameters()`` for data-parallel runs."""

    def __init__(self, model, optimizer=None, class_weights: bool = True, buckets=None, use_graph: bool = True):
        self.model, self.opt, self.buckets, self.use_graph = model, optimizer, buckets, use_graph
        dev = model.s.device
        if dev.type != "cuda":
            raise RuntimeError("abcnet_b200.TrainStep needs the model on a CUDA (sm_100) device; there is no CPU path")
        _lib.require_device()
        self.type_w = torch.tensor(ATOM_TYPE_WEIGHTS, dtype=torch.float32, device=dev) if class_weights else None
        self.params = [p for p in model.parameters() if p.requires_grad]
        if buckets is None:
            for p in self.params:
                if p.grad is None:
                    p.grad = torch.zeros_like(p)
        self.graph = None
        self.launches_per_step = 0
        self._x = self._tg = None
        self.loss = torch.zeros((), dtype=torch.float64, device=dev)
        self.parts = torch.zeros(8, dtype=torch.float64, device=dev)
        self._opt_in_graph = optimizer is not None and bool(optimizer.defaults.get("capturable", False))
        self._det = None                                   # torch.are_deterministic_algorithms_enabled() when the graph was captured

    # ------------------------------------------------------------------ the enqueued work
    def _sink(self, p, g):
        if not p.requires_grad:
            return
        if self.buckets is not None:
            p.grad.add_(g.to(p.grad.dtype).view_as(p.grad))
            self.buckets.grad_ready(p)
        else:
            p.grad.copy_(g.view_as(p.grad))

    def _enqueue(self, x, targets, with_opt):
        m = self.model
        eng = m._train_engine()
        if self.buckets is not None:
            self.buckets.zero()
        outs = eng.forward(x)
        if p8_loss_supported(outs) and not os.environ.get("ABCNET_LOSS_FP32"):
            # the loss writes the (unscaled) gradient straight into the bf16 P8 operands of the head gradient GEMMs
            p8 = eng.head_grad_buffers()
            total, parts, ds, head_scale = loss_forward_p8(m.s, self.type_w, list(targets), outs, *p8)
            dlogits = None
        else:                                              # other head lists: fp32 gradient maps + one conversion pass per head
            p8 = None
            total, parts, ds, dlogits, head_scale = loss_forward_backward(m.s, self.type_w, list(targets), outs, scaled=False)
        self.loss.copy_(total)
        self.parts.copy_(parts)
        self._sink(m.s, ds.to(m.s.dtype))
        eng.backward(dlogits, self._sink, head_scale=head_scale, p8=p8)
        if self.buckets is not None:
            self.buckets.finish()
        if with_opt and self.opt is not None:
            self.opt.step()

    # ------------------------------------------------------------------ public
    @torch.no_grad()
    def __call__(self, x, targets: Sequence[torch.Tensor]):
        if not self.model.training:
            raise RuntimeError("TrainStep: call model.train() first")
        self.model.invalidate_packed()        # a graph replay updates weights / running statistics behind torch's version counters
        if not self.use_graph:
            self._enqueue(x, targets, True)
            return self.loss.clone()
        if self.graph is not None and self._det != torch.are_deterministic_algorithms_enabled():
            self.graph = None                              # the other reduction mode is a different set of kernels: re-capture
        if self.graph is not None and (x.shape != self._x.shape or x.dtype != self._x.dtype):
            # e.g. the last, partial batch of a DataLoader without drop_last (the reference's loaders, train.py:43-46): run
            # it eagerly through the same kernels; the graph of the regular batch shape stays valid (its buffers are keyed
            # by shape inside the engine and are re-created on the next regular call only if the eager pass replaced them)
            self._enqueue(x, targets, True)
            self.graph = None                              # engine buffers were re-shaped: re-capture on the next regular batch
            return self.loss.clone()
        if self.graph is None:
            self._capture(x, targets)
        else:
            if x.data_ptr() != self._x.data_ptr():
                self._x.copy_(x, non_blocking=True)
            for dst, src in zip(self._tg, targets):
                if src.data_ptr() != dst.data_ptr():
                    dst.copy_(src, non_blocking=True)
        if self._opt_in_graph and hasattr(self.opt, "sync_hyperparams"):
            self.opt.sync_hyperparams()                    # lr edits of param_groups reach the device before the replay
        self.graph.replay()
        if self.opt is not None and not self._opt_in_graph:
            self.opt.step()
        return self.loss.clone()                           # a fresh tensor per step: callers may collect the returned losses

    def _capture(self, x, targets):
        self._det = torch.are_deterministic_algorithms_enabled()
        # static input buffers; the first batch is also used for the warm-up iterations (parameters are restored after)
        self._x = x.clone()
        self._tg = [t.clone() for t in targets]
        state = [p.detach().clone() for p in self.model.parameters()]
        bufs = [b.detach().clone() for b in self.model.buffers()]
        opt_in = self._opt_in_graph
        opt_state = {}
        if opt_in:                                         # optimiser state must exist before capture (lazy init is not replayable)
            opt_state = {p: {k: (v.clone() if torch.is_tensor(v) else v) for k, v in st.items()} for p, st in self.opt.state.items()}
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                      # warm-up outside capture: lazy attribute / allocator work
            for _ in range(2):
                self._enqueue(self._x, self._tg, opt_in)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.no_grad():                              # undo the BatchNorm running-statistics updates of the warm-up
            for p, s in zip(self.model.parameters(), state):
                p.copy_(s)
            for b, s in zip(self.model.buffers(), bufs):
                b.copy_(s)
            if opt_in:                                     # ... and the optimiser's moments / step counters
                for p, st in self.opt.state.items():
                    for k, v in st.items():
                        if torch.is_tensor(v):
                            if p in opt_state:
                                v.copy_(opt_state[p][k])
                            else:
                                v.zero_()
        self.graph = torch.cuda.CUDAGraph()
        l0 = _lib.launch_count()
        with torch.cuda.graph(self.graph):
            self._enqueue(self._x, self._tg, self._opt_in_graph)
        self.launches_per_step = _lib.launch_count() - l0      # kernels of this library inside one replay


def make_optimizer(model, lr: float = 2.5e-4, weight_decay: float = 1e-8, capturable: bool = True, fused: bool = True):
    """The reference's optimiser (``train.py:55``: Adam, lr 2.5e-4, L2 1e-8), graph-capturable. ``fused=True`` (default):
    ``abcnet_b200.FusedAdam`` -- one kernel launch for all parameters; ``fused=False``: ``torch.optim.Adam`` (foreach)."""
    params = [p for p in model.parameters() if p.requires_grad]
    if fused:
        from .optim import FusedAdam
        return FusedAdam(params, lr=lr, weight_decay=weight_decay)
    return torch.optim.Adam(params, lr=lr, weight_decay=weight_decay, capturable=capturable, foreach=True)
