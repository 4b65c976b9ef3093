"""CUDA-graph capture of the training step (forward + loss + backward).

A ConvCNP meta-batch step is ~50 kernels of 10-50 us each: eager PyTorch dispatch (autograd Function bookkeeping + one
ctypes call per kernel) costs about as much host time as the kernels cost device time, so the GPU idles between launches.
``GraphedStep`` records the whole step once per input-shape signature into a ``torch.cuda.CUDAGraph`` and replays it:
one host call per step, kernels back to back on the device.

    step = GraphedStep(model, criterion)            # optionally flat=FlatGradients(model, process_group)
    loss = step(X_cntxt, Y_cntxt, X_trgt, Y_trgt)   # gradients are in p.grad (views of step.flat.flat) afterwards
    optimizer.step()

What is captured: ``flat.zero_()``, ``model(...)``, ``criterion(...)``, ``loss.backward()`` (and, when the one-kernel NVLink
all-reduce ``parallel.P2PAllReduce`` is set up, the flat-gradient all-reduce).  What stays outside: the host->device copies of
the inputs into the graph's static buffers, the NCCL flat-gradient all-reduce otherwise (``ReduceOp.AVG`` right after the
replay), the optimizer, and the host side of the asynchronous [-1, 1] range validation (``_validate_inputs`` only launches the
check kernel while capturing; the flag is read back after every replay).

Constraints (the usual ones of whole-network capture): shapes are static per graph -- a new (n_cntxt, n_trgt, batch)
signature records a new graph (LRU cache of ``max_graphs``); Python-side control flow is frozen at capture (number of
latent samples, train/eval mode -- the mode is part of the signature); the returned loss is a static tensor that the
next replay overwrites.
"""
from collections import OrderedDict

import torch

from . import ops
from .parallel import FlatGradients

__all__ = ["GraphedStep", "PipelinedStep"]


class _Entry:
    __slots__ = ("graph", "inputs", "loss", "launches")


class GraphedStep:
    def __init__(self, model, criterion, flat=None, n_warmup=2, max_graphs=8):
        self.model, self.criterion = model, criterion
        if any(getattr(m, "_npf_sync_group", None) is not None for m in model.modules()):
            raise NotImplementedError("GraphedStep: synchronised BatchNorm (parallel.sync_batchnorm_) issues collectives from the autograd "
                                      "thread inside backward; run that configuration eagerly")
        self.flat = flat if flat is not None else FlatGradients(model)
        self.n_warmup, self.max_graphs = n_warmup, max_graphs
        # where the gradient all-reduce of a multi-GPU step runs: the one-kernel NVLink all-reduce (parallel.P2PAllReduce) is
        # recorded into the graph (0.758 vs 0.762 ms at N=2 on B200, profiles/r2/allreduce_placement.md); the NCCL fallback runs
        # right after the replay on the caller's stream (no difference measured either way)
        self.allreduce_in_graph = getattr(self.flat, "p2p", None) is not None
        self._graphs = OrderedDict()
        self._side = None

    # the eager body; also what gets recorded
    def _body(self, xc, yc, xt, yt):
        self.flat.zero_()
        out = self.model(xc, yc, xt, yt)
        loss = self.criterion(out, yt)
        if self.model.training:        # an eval-mode signature replays forward + loss only
            loss.backward()
            if self.allreduce_in_graph:
                # multi-GPU: the flat-gradient all-reduce recorded into the step (NCCL collectives are capturable): a replay
                # then has no host-side launch after the backward
                self.flat.all_reduce_mean()
        return loss.detach()

    def _signature(self, tensors):
        """Everything a recorded graph froze: mode, input shapes, the induced grid (``set_extrapolation`` changes its
        length), the number of latent samples, the arithmetic mode, and the parameter / gradient storage the kernels
        were given pointers to (``FlatAdam`` re-points ``p.data``; a replay after that would train stale storage)."""
        m = self.model
        xi = getattr(m, "X_induced", None)
        extra = (None if xi is None else (xi.data_ptr(), tuple(xi.shape)), getattr(m, "n_z_samples_train", None), getattr(m, "n_z_samples_test", None),
                 ops.get_precision(), hash(tuple(p.data_ptr() for p in self.flat.params)), self.flat.flat.data_ptr())
        return (m.training,) + tuple((tuple(t.shape), t.dtype) for t in tensors) + extra

    def _capture(self, sig, tensors):
        dev = next(self.model.parameters()).device
        e = _Entry()
        e.inputs = [torch.empty(t.shape, dtype=t.dtype, device=dev) for t in tensors]
        for d, s in zip(e.inputs, tensors):
            d.copy_(s, non_blocking=True)
        # warm-up on a side stream (lazy one-time initialisation inside the library, allocator pools); the running
        # statistics / step counters it advances are restored so that capture has no side effect on the model
        saved = [(b, b.clone()) for b in self.model.buffers()]
        # warm-up AND capture run on one dedicated side stream: autograd nodes that outlive a backward pass (the parameters'
        # gradient accumulators) remember the stream they were created on, and the engine joins that stream with the caller's
        # at the end of backward() -- a join with a stream outside the capture would be an illegal cross-stream dependency
        if self._side is None:
            self._side = torch.cuda.Stream(device=dev)
        side = self._side
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(self.n_warmup):
                self._body(*e.inputs)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.model.validate_now() if hasattr(self.model, "validate_now") else None
        e.graph = torch.cuda.CUDAGraph()
        n0 = ops.launch_count()
        with torch.cuda.graph(e.graph, stream=side):
            e.loss = self._body(*e.inputs)
        e.launches = ops.launch_count() - n0
        with torch.no_grad():
            for b, v in saved:
                b.copy_(v)
        self._graphs[sig] = e
        while len(self._graphs) > self.max_graphs:
            self._graphs.popitem(last=False)
        return e

    def __call__(self, X_cntxt, Y_cntxt, X_trgt, Y_trgt):
        tensors = (X_cntxt, Y_cntxt, X_trgt, Y_trgt)
        sig = self._signature(tensors)
        e = self._graphs.get(sig)
        if e is None:
            if hasattr(self.model, "validate_now"):
                self.model.validate_now()        # a new signature: surface the previous step's range check first
            e = self._capture(sig, tensors)
        else:
            self._graphs.move_to_end(sig)
        for d, s in zip(e.inputs, tensors):
            if d.data_ptr() != s.data_ptr():
                d.copy_(s, non_blocking=True)
        e.graph.replay()
        if hasattr(self.model, "_after_graph_replay"):
            self.model._after_graph_replay()
        if not self.allreduce_in_graph and self.model.training:
            self.flat.all_reduce_mean()
        self.last_launches = e.launches
        return e.loss

    def static_inputs(self, X_cntxt, Y_cntxt, X_trgt, Y_trgt):
        """The graph's own input buffers for this signature (write the next batch into them to skip the copies)."""
        tensors = (X_cntxt, Y_cntxt, X_trgt, Y_trgt)
        sig = self._signature(tensors)
        e = self._graphs.get(sig) or self._capture(sig, tensors)
        return tuple(e.inputs)


class PipelinedStep:
    """Host-side input / result pipeline around a ``GraphedStep`` for batches that start in (pinned) host memory:

        pipe = PipelinedStep(step)
        for batch in loader:                       # dict(X_cntxt=, Y_cntxt=, X_trgt=, Y_trgt=) of pinned CPU tensors
            prev_loss = pipe.submit(batch)         # float loss of the PREVIOUS step (None for the first call)
        last_loss = pipe.drain()

    Every step still does its own host->device copy of the inputs and its own device->host read of the loss; what changes is *when*:
    the copy of step i+1 runs on a side stream into a staging buffer while step i's graph replays (a 2 us device-to-device copy
    moves it into the graph's static inputs), and the loss of step i is read back while step i+1 runs, so the GPU never idles on
    PCIe latency or on the host's ``.item()`` round trip.  Gradients of step i are complete when ``submit`` of step i returns in
    stream order (run the optimizer on the same stream as usual)."""

    def __init__(self, step):
        self.step = step
        self._copy = None
        self._stage = [None, None]
        self._h2d = [None, None]
        self._used = [None, None]
        self._loss_host = None
        self._loss_ev = [None, None]
        self._i = 0

    def _setup(self, batch, dev):
        self._copy = torch.cuda.Stream(device=dev)
        for k in range(2):
            self._stage[k] = {n: torch.empty(t.shape, dtype=t.dtype, device=dev) for n, t in batch.items()}
            self._h2d[k], self._used[k] = torch.cuda.Event(), torch.cuda.Event()
            self._loss_ev[k] = torch.cuda.Event()
        self._loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()

    def _enqueue_copy(self, batch, k, dev):
        with torch.cuda.stream(self._copy):
            if self._i >= 2:
                self._copy.wait_event(self._used[k])              # the step that last read this staging set has consumed it
            for n, t in batch.items():
                self._stage[k][n].copy_(t, non_blocking=True)
            self._h2d[k].record(self._copy)

    def submit(self, batch):
        dev = next(self.step.model.parameters()).device
        if self._copy is None:
            self._setup(batch, dev)
        k = self._i & 1
        self._enqueue_copy(batch, k, dev)
        main = torch.cuda.current_stream(dev)
        main.wait_event(self._h2d[k])
        st = self._stage[k]
        loss = self.step(st["X_cntxt"], st["Y_cntxt"], st["X_trgt"], st["Y_trgt"])     # copies into the graph's static inputs, replays
        self._used[k].record(main)
        self._loss_host[k:k + 1].copy_(loss.reshape(1), non_blocking=True)
        self._loss_ev[k].record(main)
        prev = None
        if self._i >= 1:
            self._loss_ev[k ^ 1].synchronize()
            prev = float(self._loss_host[k ^ 1])
        self._i += 1
        return prev

    def drain(self):
        if self._i == 0:
            return None
        k = (self._i - 1) & 1
        self._loss_ev[k].synchronize()
        return float(self._loss_host[k])
