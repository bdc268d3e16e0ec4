"""CUDA graphs for training.

1. `training_forward` (automatic): what `RealBasicVSR.forward` runs when gradients are wanted.  The reference's `train.py`
   issues ~2 000 launches per micro-step from Python; on 64x64 patches the GPU finishes them in 33 ms while the host needs
   36 - 60 ms to issue them, depending on the box.  After a few eager calls with the same input shape the forward and the
   backward of the model are captured once (the `torch.cuda.make_graphed_callables` recipe) and replayed: the caller's loop - autocast,
   GradScaler, gradient accumulation, clipping, optimizer, DDP wrapper - stays what it is.  `VSRB_TRAIN_GRAPHS=0` switches it
   off (`VSRB_TRAIN_GRAPHS_DDP=0`: only under torch.distributed); it is not used inside someone else's capture.
2. `GraphedTrainStep` (opt-in): whole-step capture for training loops that can afford static shapes.

The reference's `train.py` launches ~1 500 kernels per step from Python; on 64x64 patches the B200 finishes them faster than
the host can issue them (cfg4: 48 ms eager vs 43 ms of GPU work).  Every launch of libvsrb200.so is stream-ordered and
allocation-free, so forward + backward + gradient clipping + optimizer step capture into ONE graph with torch's standard
whole-network recipe; `GraphedTrainStep` packages that recipe.  Single GPU (or one graph per DDP rank with
`torch.distributed` collectives outside the graph is NOT handled here).

    step = GraphedTrainStep(model, optimizer, loss_fn, example_inputs=(lr, hr), clip_grad_norm=1.0)
    for lr, hr in loader:
        loss = step(lr, hr)          # copies the batch into the graph's static buffers and replays

`optimizer` must have been built with `capturable=True` (torch.optim.Adam / AdamW).  `loss_fn(outputs, *targets)` gets the
model's outputs and the remaining inputs.
"""
from __future__ import annotations

import os
import warnings
import weakref
from typing import Callable, Dict, Optional, Sequence

import torch

TRAIN_GRAPHS = os.environ.get("VSRB_TRAIN_GRAPHS", "1") == "1"
# Under torch.distributed (DDP): the parameters still receive their gradients through their own AccumulateGrad nodes, so
# DDP's hooks fire as usual - all buckets after the backward graph instead of interleaved with it (12 MB of gradients:
# tens of microseconds over NVLink).  The capture runs in thread-local error mode: NCCL's watchdog thread polls events.
TRAIN_GRAPHS_DDP = os.environ.get("VSRB_TRAIN_GRAPHS_DDP", "1") == "1"
TRAIN_GRAPH_AFTER = 3          # eager calls (with a backward) of one (shape, flags) key before the capture
TRAIN_GRAPH_KEYS = 2           # captured call patterns kept per model (each owns the activations its backward needs)
_auto_off = 0                  # > 0 while GraphedTrainStep warms up / captures its own whole-step graph


class _TrainBody(torch.nn.Module):
    """The differentiable forward as a module of its own, so that `make_graphed_callables` finds the parameters."""

    def __init__(self, model):
        super().__init__()
        self.model = model

    def forward(self, lr):
        from . import autograd as AG
        return AG.realbasicvsr(self.model, lr, write_back=False)


class _TrainEntry:
    def __init__(self, model, key):
        self.model_ref, self.key, self.backwards, self.graphed, self.failed = weakref.ref(model), key, 0, None, False

    def saw_backward(self, _grad):
        self.backwards += 1               # (tensor hook on an eager call's `sr`: this call pattern does train)


_train_entries: Dict[int, dict] = {}


def graphed_patterns(model) -> int:
    """How many call patterns of `model` currently replay from CUDA graphs (tests, bench.py)."""
    t = _train_entries.get(id(model))
    return 0 if t is None or t["model"]() is not model else sum(e.graphed is not None for e in t["by_key"].values())


class _GraphedTraining:
    """Forward graph + backward graph of the model's differentiable forward for one input shape.

    Same recipe as `torch.cuda.make_graphed_callables`, with one difference that matters for loops on the legacy default
    stream: the capture differentiates with respect to fresh leaf ALIASES of the parameters (`p.detach().requires_grad_()`,
    same storage, same version counter), substituted through `torch.func.functional_call`.  The parameters' own
    AccumulateGrad nodes - created by earlier eager iterations on the default stream and still alive while the caller holds
    last iteration's `loss` - would otherwise make the capturing stream synchronise with the legacy stream, which CUDA refuses
    ("operation would make the legacy stream depend on a capturing blocking stream")."""

    def __init__(self, model, lr: torch.Tensor, warmup: int = 2):
        from . import functional as VF
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
        self.params = [p for _, p in named]
        aliases = [p.detach().requires_grad_() for p in self.params]
        amap = {"model." + n: a for (n, _), a in zip(named, aliases)}
        body = _TrainBody(model)
        body.train(model.training)

        def run(x):
            return torch.func.functional_call(body, amap, (x,))
        self.static_in = lr.detach().clone()
        cur = torch.cuda.current_stream(lr.device)
        side = torch.cuda.Stream(device=lr.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):
                out = run(self.static_in)
                torch.autograd.grad(out, aliases, [torch.zeros_like(o) for o in out], allow_unused=True)
                del out
        cur.wait_stream(side)
        torch.cuda.synchronize(lr.device)
        pool = torch.cuda.graph_pool_handle()
        self.fwd, self.bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        VF.REPACK_IN_CAPTURE = True
        try:
            with torch.cuda.graph(self.fwd, pool=pool, capture_error_mode="thread_local"):
                self.static_out = run(self.static_in)
            self.static_gout = [torch.zeros_like(o) for o in self.static_out]
            with torch.cuda.graph(self.bwd, pool=pool, capture_error_mode="thread_local"):
                self.static_gin = torch.autograd.grad(self.static_out, aliases, self.static_gout, allow_unused=True)
        finally:
            VF.REPACK_IN_CAPTURE = False
        self.static_out = tuple(o.detach() for o in self.static_out)       # (drops the captured autograd graph)
        self.pending = False

    def __call__(self, lr: torch.Tensor):
        return _ReplayFn.apply(self, lr, *self.params)


class _ReplayFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, entry, lr, *params):
        entry.static_in.copy_(lr)
        entry.fwd.replay()
        ctx.entry = entry
        entry.pending = True              # the saved activations now belong to THIS call until its backward has run
        return tuple(o.detach() for o in entry.static_out)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *gouts):
        e = ctx.entry
        for g, sg in zip(gouts, e.static_gout):
            if g is None:
                sg.zero_()
            elif g.data_ptr() != sg.data_ptr():
                sg.copy_(g)
        e.bwd.replay()
        e.pending = False
        # CLONES: AccumulateGrad may adopt an incoming gradient as `p.grad` without copying; a view of the graph's static
        # buffer would then be overwritten by the next replay - with gradient accumulation the first micro-step's gradient
        # would be lost and the second counted twice (12 MB of parameters: the copies cost microseconds)
        return (None, None) + tuple(None if g is None else g.clone() for g in e.static_gin)


def _capture_training(model, lr: torch.Tensor):
    global _auto_off
    _auto_off += 1                        # the body's own calls of the model must run the eager path
    try:
        if torch.is_autocast_enabled("cuda"):             # the caller's autocast, minus its weight-cast cache (not capturable)
            with torch.autocast("cuda", dtype=torch.get_autocast_dtype("cuda"), cache_enabled=False):
                return _GraphedTraining(model, lr)
        return _GraphedTraining(model, lr)
    finally:
        _auto_off -= 1


def training_forward(model, lr: torch.Tensor):
    """(sr, lq) with gradients; replays a captured forward / backward once the call pattern has settled."""
    from . import autograd as AG
    from . import ops
    dist_on = torch.distributed.is_available() and torch.distributed.is_initialized() and not TRAIN_GRAPHS_DDP
    if (not TRAIN_GRAPHS or _auto_off or dist_on or lr.requires_grad or lr.dtype != torch.float32 or not lr.is_contiguous()
            or ops.PROFILE is not None or torch.cuda.is_current_stream_capturing()):
        return AG.realbasicvsr(model, lr)
    params = list(model.parameters())
    key = (tuple(lr.shape), str(lr.device), model.training, torch.is_autocast_enabled("cuda"),
           tuple(p.requires_grad for p in params), tuple(p.data_ptr() for p in params),
           torch.are_deterministic_algorithms_enabled())      # the deterministic kernels are a different graph
    table = _train_entries.get(id(model))
    if table is None or table["model"]() is not model:
        table = {"model": weakref.ref(model), "by_key": {}}
        _train_entries[id(model)] = table
        weakref.finalize(model, _train_entries.pop, id(model), None)
    by_key = table["by_key"]
    e = by_key.pop(key, None)
    if e is None:
        e = _TrainEntry(model, key)
        while len(by_key) >= TRAIN_GRAPH_KEYS:            # (a training and an evaluation pattern; dicts keep insertion order)
            by_key.pop(next(iter(by_key)))
    by_key[key] = e                                       # most recently used last
    if e.graphed is None and not e.failed and e.backwards >= TRAIN_GRAPH_AFTER:
        try:
            e.graphed = _capture_training(model, lr)
        except Exception as exc:          # keep training eagerly rather than fail the step
            e.failed = True
            warnings.warn(f"vsrlab_b200: training-graph capture failed ({type(exc).__name__}: {exc}); staying eager", RuntimeWarning)
    if e.graphed is None or e.graphed.pending:
        # (a second forward before the first one's backward - two generator passes per step - must not overwrite the
        # activations the graph saved for that backward: eager.  Patterns that never backpropagate - an evaluation loop that
        # leaves grad mode on - are never captured: only eager calls whose `sr` received a gradient count.)
        sr, lq = AG.realbasicvsr(model, lr)
        if e.graphed is None and not e.failed and sr.requires_grad:
            sr.register_hook(e.saw_backward)
        return sr, lq
    sr, lq = e.graphed(lr)
    with torch.no_grad():
        lr.copy_(lq)                      # the reference refines its input in place (realbasicvsr.py:26-29)
    return sr, lq


class GraphedTrainStep:
    def __init__(self, model: torch.nn.Module, optimizer: torch.optim.Optimizer, loss_fn: Callable,
                 example_inputs: Sequence[torch.Tensor], clip_grad_norm: Optional[float] = None,
                 autocast_dtype: Optional[torch.dtype] = torch.bfloat16, warmup: int = 3):
        if not all(g.get("capturable", False) for g in optimizer.param_groups):
            raise ValueError("GraphedTrainStep needs an optimizer created with capturable=True")
        self.model, self.opt, self.loss_fn, self.clip, self.dtype = model, optimizer, loss_fn, clip_grad_norm, autocast_dtype
        global _auto_off
        _auto_off += 1                                    # this class captures the whole step itself
        try:
            self._build(example_inputs, warmup)
        finally:
            _auto_off -= 1

    def _build(self, example_inputs, warmup):
        self.static_in = [t.clone() for t in example_inputs]
        self.stream = torch.cuda.Stream(device=self.static_in[0].device)
        self.warmup = warmup
        self._graphs = {}                                 # torch.are_deterministic_algorithms_enabled() -> (graph, loss)
        self._capture(update=True)

    def _capture(self, update: bool):
        """Warm up and capture the step for the current value of the deterministic flag.  `update`: the warm-up steps are
        real training steps (construction); otherwise they run forward and backward only and discard the gradients, so a
        capture for the other flag value in the middle of a run changes neither the parameters nor the optimizer state."""
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):              # warm-up on the capture stream (also where the grad accumulators live)
            for _ in range(self.warmup):
                self.opt.zero_grad(set_to_none=True)
                self._body(update)
        torch.cuda.current_stream().wait_stream(self.stream)
        torch.cuda.synchronize()
        self.opt.zero_grad(set_to_none=True)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            self.static_loss = self._body()
        self._graphs[torch.are_deterministic_algorithms_enabled()] = (self.graph, self.static_loss)

    def _body(self, update: bool = True) -> torch.Tensor:
        x = self.static_in[0].clone()                     # the model refines its input in place (reference contract)
        if self.dtype is not None:
            with torch.autocast("cuda", dtype=self.dtype):
                out = self.model(x)
        else:
            out = self.model(x)
        loss = self.loss_fn(out, *self.static_in[1:])
        loss.backward()
        if not update:
            return loss.detach()
        if self.clip is not None:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.clip)
        self.opt.step()
        return loss.detach()

    def __call__(self, *inputs: torch.Tensor) -> torch.Tensor:
        for dst, src in zip(self.static_in, inputs):
            dst.copy_(src, non_blocking=True)
        det = torch.are_deterministic_algorithms_enabled()
        if det not in self._graphs:                       # the flag changed since the capture: capture the other kernels too
            global _auto_off
            _auto_off += 1
            try:
                self._capture(update=False)
            finally:
                _auto_off -= 1
        self.graph, self.static_loss = self._graphs[det]
        self.graph.replay()
        return self.static_loss
