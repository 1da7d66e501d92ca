"""Whole-training-step CUDA graph for ``UnetWrapper.training_step`` (models/wrapper.py:117-162 of the reference).

One GAN step is ~520 kernel launches of 5-250 us each (implicit-GEMM convs, BatchNorm / activation streams, the
fused Adam, a few torch scalar ops): issued from Python the host is the bottleneck for ~10 % of the step (measured
with the CUPTI timeline: 1.3 ms of GPU idle time per 12.5 ms step).  ``StepGraph`` captures the *entire* step --
both forwards, both backwards, the gradient all-reduces, both optimizer steps and the logged metrics -- once per
input shape and replays it with one ``cudaGraphLaunch``:

* the first ``warmup`` calls per shape run eagerly (allocations, lazily built weight packs, optimizer state);
* the capture call records the step on static input buffers without executing it, then the graph is replayed;
* every later call copies the batch into the static buffers, replays, and logs clones of the static outputs.

What makes the step capturable: the library never synchronises or allocates, FusedAdam keeps its step counter and
bias-correction scalars on the device (``pai_adam_prepare``), BatchNorm bookkeeping is device-side, and the
orchestration holds no data-dependent Python control flow.  The graph bakes in pointers (parameters, optimizer state,
weight packs) and scalars (lr, betas, eps, ``requires_grad`` pattern): a cheap signature check before every replay
drops the graph and re-captures when any of them changed (``load_state_dict``, ``.to()``, a new learning rate).
"""
from __future__ import annotations

import gc

import torch

from . import lib


class _Entry:
    def __init__(self):
        self.eager_calls = 0
        self.graph = None
        self.static_x = self.static_t = None
        self.outputs = []          # [(name, static tensor)] in logging order
        self.signature = None
        self.launches = 0


class StepGraph:
    def __init__(self, module, warmup: int = 3):
        self.module = module
        self.warmup = max(1, int(warmup))
        self.entries = {}
        self.replays = 0

    # ---- what the graph bakes in ---------------------------------------------------------------------------
    def _signature(self):
        m = self.module
        sig = []
        for p in m.parameters():
            sig.append((p.data_ptr(), p.requires_grad))
            packs = p.__dict__.get("_pai_packs")
            if packs:
                sig.extend(ent[1].data_ptr() for ent in packs.values())
        for b in m.buffers():
            sig.append(b.data_ptr())
        opts = m.optimizers()
        for opt in (opts if isinstance(opts, (list, tuple)) else [opts]):
            for group in opt.param_groups:
                sig.append((float(group["lr"]), tuple(group["betas"]), float(group["eps"])))
            for st in opt.state.values():
                if "exp_avg" in st:
                    sig.append(st["exp_avg"].data_ptr())
        return tuple(sig)

    def _drop_lazy_packs(self):
        """Forgets every weight pack that the optimizer does NOT refresh in place (thin-layer / auxiliary packs and
        all packs of the layer-node models): FusedAdam drops them after each update and the next forward rebuilds
        them.  A pack built eagerly before the capture would be baked into the graph as a pointer to memory that the
        captured optimizer step releases -- the replays would read weights frozen at capture time (or freed memory).
        Dropping them first makes the capture rebuild each of them INSIDE the graph, from the live parameters, into
        graph-pool memory, at every replay."""
        from . import engine
        for p in self.module.parameters():
            p.__dict__.pop("_pai_aux", None)
            if p.__dict__.get("_pai_packs") and engine.fused_pack_targets(p) is None:
                p.__dict__.pop("_pai_packs", None)

    def _capture(self, ent: _Entry, x, target, batch_idx):
        m = self.module
        ent.static_x, ent.static_t = x.clone(), target.clone()
        self._drop_lazy_packs()
        ent.signature = self._signature()
        torch.cuda.synchronize()
        # A discarded module with its StepGraph is a reference cycle that only the cyclic garbage collector frees, CUDA
        # graphs included; destroying a graph while this one is being captured invalidates the capture.  So dead cycles
        # are collected now and the collector stays off until the capture ends.
        gc.collect()
        gc_enabled = gc.isenabled()
        gc.disable()
        sink = []
        m.__dict__["_pai_log_sink"] = sink           # _training_step_eager logs into it instead of calling self.log
        launches0 = lib.launches
        graph = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(graph):
                m._training_step_eager((ent.static_x, ent.static_t), batch_idx)
        finally:
            if gc_enabled:
                gc.enable()
            m.__dict__.pop("_pai_log_sink", None)
        ent.launches = lib.launches - launches0
        lib.launches = launches0                     # nothing ran during capture
        ent.outputs = list(sink)
        ent.graph = graph
        if self._signature() != ent.signature:       # e.g. a pack built for the first time inside the capture
            ent.signature = self._signature()

    def __call__(self, batch, batch_idx):
        m = self.module
        x, target = batch
        if not (x.is_cuda and target.is_cuda):
            return m._training_step_eager(batch, batch_idx)
        key = (tuple(x.shape), x.dtype, tuple(target.shape), target.dtype, x.device, m.training)
        ent = self.entries.get(key)
        if ent is None:
            ent = self.entries[key] = _Entry()
        if ent.graph is not None and self._signature() != ent.signature:
            self.entries[key] = ent = _Entry()       # pointers / hyper-parameters moved: warm up and capture again
        if ent.graph is None:
            if ent.eager_calls < self.warmup:
                ent.eager_calls += 1
                return m._training_step_eager(batch, batch_idx)
            self._capture(ent, x, target, batch_idx)
        ent.static_x.copy_(x, non_blocking=True)
        ent.static_t.copy_(target, non_blocking=True)
        ent.graph.replay()
        self.replays += 1
        lib.launches += ent.launches
        for name, v in ent.outputs:               # static graph outputs -> the module's own log (Lightning's or the shim's)
            m.log(name, v.clone(), prog_bar=True)
        return None
