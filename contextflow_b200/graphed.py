"""CUDA-graph replay of the log-density forward.

One `log_prob` is 150-200 kernel launches, most of them microseconds long; issued one by one from Python the launch
overhead (ctypes call + torch allocation + driver launch, ~10-20 us each) exceeds the device time of the small kernels and
the GPU idles between them.  `GraphedLogProb` captures the whole forward for a fixed input shape once (torch.cuda.CUDAGraph
over the stream the C-ABI kernels are launched on) and replays it per batch: inputs are copied into the capture's static
buffers (a pinned host tensor is copied host->device straight into them), one `cudaGraphLaunch` runs the step, the (B, M)
log-probabilities are returned as a fresh tensor.  The RNG draws inside the path (torch.rand / torch.randn) are graph-safe:
torch advances the Philox offset on every replay.

Capture requirements met by the path: no host synchronisation inside a forward (ActNorm's one-time initialisation read happens
in the eager warm-up), no host memory copies inside the library, every buffer allocated through torch's graph pool.
"""
from __future__ import annotations

import contextlib
import gc
import operator
import weakref

import torch
from torch._utils import _flatten_dense_tensors, _unflatten_dense_tensors

from . import _cabi

_version_of = operator.attrgetter('_version')


class _Entry:
    __slots__ = ('graph', 'x', 'ctx', 'out', 'launches', 'signature', 'device', 'host_draws')


class GraphedLogProb:
    def __init__(self, model, warmup: int = 2):
        self.model, self.warmup = model, max(1, warmup)
        self._entries = {}
        self._pool = None
        self._tensors = None

    def _device(self):
        """The model's device (the reference places it with .to('cuda:{gpu}') and never calls set_device, model.py:170,285)."""
        for p in self.model.parameters():
            if p.is_cuda:
                return p.device
        return torch.device('cuda', torch.cuda.current_device())

    def _signature(self):
        """Changes whenever a parameter / buffer is written in place (optimizer step, load_state_dict, ActNorm initialisation) or moved
        (.to(), .double()): the layers repack weights on the host side keyed on these versions, so a captured graph is only valid for
        the signature it was captured under.  Cost matters at small batches (reference default B = 256: a replay is ~0.5 ms of device
        time): the tensor list is cached (rebuilt when the module tree is re-applied, see FlowSequential._apply) and only the version
        counters are read per call -- ~0.1 ms for the ~1200 tensors of cfg2 instead of 7 ms for a state_dict() walk."""
        ts = self._tensors
        if ts is None:
            ts = self._tensors = list(self.model.parameters()) + list(self.model.buffers())
            self._ptrs = hash(tuple(t.data_ptr() for t in ts))
        return hash(tuple(map(_version_of, ts))) ^ self._ptrs

    def invalidate(self):
        """Forget the cached tensor list and every captured graph (the module tree was moved / cast / restructured)."""
        self._tensors = None
        self._entries.clear()

    def _capture(self, x, ctx, device):
        with torch.cuda.device(device):
            return self._capture_on(x, ctx, device)

    def _capture_on(self, x, ctx, device):
        e = _Entry()
        e.device = device
        e.x = torch.empty(x.shape, device=device, dtype=x.dtype)
        e.ctx = None if ctx is None else torch.empty(ctx.shape, device=device, dtype=ctx.dtype)
        e.x.copy_(x)
        if ctx is not None:
            e.ctx.copy_(ctx)
        # the eager warm-up and the capture consume random numbers; the generators are put back afterwards so that the FIRST replay sees
        # exactly the draws an eager call at this point would have seen (same seed => same noise as the eager path / the reference)
        from . import rng
        cpu_state, cuda_state = torch.get_rng_state(), torch.cuda.get_rng_state(device)
        cur = torch.cuda.current_stream(device)
        side = torch.cuda.Stream(device)
        side.wait_stream(cur)
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(self.warmup):                       # eager: ActNorm init, weight repacking, attribute setup
                self.model.log_prob_eager(e.x, e.ctx)
        cur.wait_stream(side)
        torch.cuda.synchronize(device)
        e.graph = torch.cuda.CUDAGraph()
        l0 = _cabi.launch_count()
        del rng._capture_host_draws[:]
        # explicit capture stream on THIS device: torch.cuda.graph's default capture stream is created once per process, on whichever
        # device was current at the first capture, and would drag captures of replicas on other GPUs (multigpu.py) onto that device
        with torch.no_grad(), torch.cuda.graph(e.graph, pool=self._pool, stream=side):
            e.out = self.model.log_prob_eager(e.x, e.ctx)
        e.launches = _cabi.launch_count() - l0
        e.host_draws = list(rng._capture_host_draws)
        del rng._capture_host_draws[:]
        torch.set_rng_state(cpu_state); torch.cuda.set_rng_state(cuda_state, device)
        if self._pool is None:
            self._pool = e.graph.pool()
        e.signature = self._signature()
        return e

    def entry(self, x, ctx):
        key = (tuple(x.shape), x.dtype, None if ctx is None else (tuple(ctx.shape), ctx.dtype))
        e = self._entries.get(key)
        if e is not None and e.signature != self._signature():    # weights changed since capture (training step, load_state_dict)
            e = None
        if e is None:
            dev = x.device if x.is_cuda else self._device()
            e = self._entries[key] = self._capture(x, ctx, dev)
        return e

    def launches_per_replay(self, x, ctx):
        return self.entry(x, ctx).launches

    def __call__(self, x, ctx=None, clone: bool = True):
        """x / ctx may live on the device or in (pinned) host memory; returns the (B, M) log-probabilities."""
        e = self.entry(x, ctx)
        if e.device.index != torch.cuda.current_device():
            with torch.cuda.device(e.device):
                return self._replay(e, x, ctx, clone)
        return self._replay(e, x, ctx, clone)

    @staticmethod
    def _replay(e, x, ctx, clone):
        e.x.copy_(x, non_blocking=True)
        if ctx is not None:
            e.ctx.copy_(ctx, non_blocking=True)
        for buf in e.host_draws:                               # rng 'host' mode: the CPU-generator draws of this forward (uniform.py:32)
            buf.copy_(torch.rand(buf.shape, dtype=buf.dtype))
        e.graph.replay()
        return e.out.clone() if clone else e.out

    def stream(self, batches, outs, post=None):
        """Throughput mode for host-resident data: `batches` yields (x, ctx) pinned host tensors of one shape, `outs[i]` is the
        pinned host tensor that receives batch i's (B, M) log-probabilities.  The host-to-device copy of batch i+1 runs on a copy
        stream while the captured graph of batch i replays (two device staging buffers); the device-to-host copy of each result
        is queued right behind its replay.  Returns after everything has completed.  `post(logp)` (optional) maps the replay's
        output to the tensor that is copied out (e.g. the all-gather of a sharded batch)."""
        with torch.cuda.device(self._device()):
            return self._stream_on(batches, outs, post)

    def _stream_on(self, batches, outs, post):
        dev = self._device()
        comp = torch.cuda.current_stream(dev)
        copy_stream = getattr(self, '_copy_stream', None)
        if copy_stream is None:
            copy_stream = self._copy_stream = torch.cuda.Stream(dev)
        e, stage, ready, consumed = None, None, None, None
        for i, (hx, hc) in enumerate(batches):
            if e is None:
                e = self.entry(hx, hc)
                stage = [(torch.empty_like(e.x), None if e.ctx is None else torch.empty_like(e.ctx)) for _ in range(2)]
                ready = [torch.cuda.Event() for _ in range(2)]
                consumed = [torch.cuda.Event() for _ in range(2)]
                for ev in consumed:
                    ev.record(comp)
            k = i & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[k])              # staging buffer k has been drained into the graph's input
                stage[k][0].copy_(hx, non_blocking=True)
                if hc is not None:
                    stage[k][1].copy_(hc, non_blocking=True)
                ready[k].record(copy_stream)
            comp.wait_event(ready[k])
            e.x.copy_(stage[k][0], non_blocking=True)
            if hc is not None:
                e.ctx.copy_(stage[k][1], non_blocking=True)
            consumed[k].record(comp)
            for buf in e.host_draws:
                buf.copy_(torch.rand(buf.shape, dtype=buf.dtype))
            e.graph.replay()
            res = e.out if post is None else post(e.out)
            outs[i].copy_(res[:outs[i].shape[0]], non_blocking=True)
        comp.synchronize()
        return outs


_requires_grad_of = operator.attrgetter('requires_grad')
_suspended = 0          # > 0 while GraphedTrainStep warms up over a model: its log_prob calls under autograd then stay eager


@contextlib.contextmanager
def eager_training():
    """Calls of log_prob under autograd launch eagerly inside this block, whatever GraphedTrainLogProb is enabled."""
    global _suspended
    _suspended += 1
    try:
        yield
    finally:
        _suspended -= 1


@contextlib.contextmanager
def _leaf_aliases(model, params):
    """While a training entry warms up and captures, every trainable parameter of `model` is replaced by a fresh leaf over the same
    storage; yields those leaves.  The graphs read and the optimizer writes the same memory, but the capture never reaches the
    parameters' own AccumulateGrad nodes: the caller's previous step may keep them alive, bound to the stream of an eager call, and
    an autograd backward that synchronises with another stream cannot be captured."""
    leaves = {id(p): torch.nn.Parameter(p.detach()) for p in params}
    saved = [(m, k, v) for m in model.modules() for k, v in m._parameters.items() if v is not None and id(v) in leaves]
    for m, k, v in saved:
        m._parameters[k] = leaves[id(v)]
    try:
        yield [leaves[id(p)] for p in params]
    finally:
        for m, k, v in saved:
            m._parameters[k] = v


class _TrainEntry:
    __slots__ = ('fwd', 'bwd', 'x', 'ctx', 'out', 'dlogp', 'flat', 'used', 'slots', 'params', 'frozen', 'versions', 'host_draws',
                 'device', 'generation', 'waiting')


class _ReplayTrain(torch.autograd.Function):
    """Joins an entry's forward and backward graphs to the caller's autograd graph.  The trainable parameters are the inputs, so the
    backward hands autograd one gradient per parameter and the caller's loss, backward() and optimizer stay where they are."""

    @staticmethod
    def forward(ctx, e, x, c, *params):
        e.x.copy_(x, non_blocking=True)
        if c is not None:
            e.ctx.copy_(c, non_blocking=True)
        for buf in e.host_draws:                                # rng 'host' mode: the CPU-generator draws of this forward
            buf.copy_(torch.rand(buf.shape, dtype=buf.dtype))
        if e.device.index != torch.cuda.current_device():
            with torch.cuda.device(e.device):
                e.fwd.replay()
        else:
            e.fwd.replay()
        e.generation += 1
        ctx.entry, ctx.generation = e, e.generation
        e.waiting = weakref.ref(ctx)                            # this replay's activations wait for its backward
        return e.out.detach().clone()                           # the caller may edit its log-probabilities in place

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dlogp):
        e = ctx.entry
        if ctx.generation != e.generation:
            raise RuntimeError('log_prob was replayed from its CUDA graph again before this backward ran, which overwrote the activations '
                               'this backward needs.  Call backward() before the next log_prob of the same shape, or disable training '
                               'graphs with model.enable_cuda_graphs(training=False).')
        e.dlogp.copy_(dlogp)
        e.bwd.replay()
        e.waiting = None
        # one device copy of all gradients; AccumulateGrad adopts the views as .grad without copying them again
        views = _unflatten_dense_tensors(e.flat.clone(), e.used) if e.used else ()
        grads = [None] * (3 + len(e.params))
        for slot, g in zip(e.slots, views):
            grads[3 + slot] = g
        return tuple(grads)


class GraphedTrainLogProb:
    """CUDA-graph replay of `log_prob` under autograd, for a training loop that keeps its own loss, backward() and optimizer step.

    Per input shape an entry holds two graphs over static buffers: the forward (log_prob_eager under autograd, derived weights
    recomputed inside the graph: live_capture) and the backward (torch.autograd.grad of the captured log-probabilities with respect to
    the trainable parameters, written into one flat gradient buffer).  `_ReplayTrain` joins them to the caller's autograd graph.

    The first call at a key (input shapes and dtypes, model.training, which parameters require grad) runs eagerly; that call also
    performs one-time work such as ActNorm's first-batch initialisation.  The second call captures and replays.  An entry stays valid
    while no parameter or buffer has moved and no tensor that does not require grad has been written: trainable parameters are read
    live by the graphs, so optimizer steps keep it valid, while values derived from frozen tensors are cached under their versions and a
    load_state_dict forces a new eager call and capture.  MAX_ENTRIES entries are kept (e.g. the full batch and the ragged last batch),
    the oldest is dropped first."""

    MAX_ENTRIES = 2

    def __init__(self, model, warmup: int = 1):
        self.model, self.warmup = model, max(1, warmup)
        self._entries = {}
        self._seen = {}             # key -> state signature after the eager call at that key
        self._tensors = None

    def invalidate(self):
        self._tensors = None
        self._entries.clear()
        self._seen.clear()

    def _state(self):
        ts = self._tensors
        if ts is None:
            self._params = list(self.model.parameters())
            ts = self._tensors = self._params + list(self.model.buffers())
            self._ptrs = hash(tuple(t.data_ptr() for t in ts))
        return ts

    def _signature(self, frozen):
        return hash(tuple(map(_version_of, frozen))) ^ self._ptrs

    def __call__(self, x, ctx=None):
        if (_suspended or x.requires_grad or (ctx is not None and (ctx.requires_grad or not ctx.is_cuda))
                or torch.cuda.is_current_stream_capturing()):
            return self.model.log_prob_eager(x, ctx)
        from . import rng
        if rng._source is not None or rng._recorder is not None:   # replayed noise tapes / draw recording are host-driven
            return self.model.log_prob_eager(x, ctx)
        ts = self._state()
        rg = tuple(map(_requires_grad_of, self._params))
        key = (tuple(x.shape), x.dtype, x.device, None if ctx is None else (tuple(ctx.shape), ctx.dtype), self.model.training, rg)
        e = self._entries.get(key)
        if e is not None and self._signature(e.frozen) != e.versions:
            del self._entries[key]                              # weights loaded or moved: eager once more, then a new capture
            e = None
        if e is None:
            frozen = [t for t in ts if not t.requires_grad]
            params = [p for p in self._params if p.requires_grad]
            if (not params or any(p._backward_hooks or p._post_accumulate_grad_hooks for p in params)
                    or self._seen.get(key) != self._signature(frozen)):
                out = self.model.log_prob_eager(x, ctx)
                self._seen.pop(key, None)
                self._seen[key] = self._signature(frozen)
                while len(self._seen) > 4 * self.MAX_ENTRIES:
                    del self._seen[next(iter(self._seen))]
                return out
            e = self._capture(x, ctx, params, frozen)
            self._entries[key] = e
            while len(self._entries) > self.MAX_ENTRIES:
                del self._entries[next(iter(self._entries))]
        elif (e.waiting is not None and e.waiting() is not None) or any(p._backward_hooks or p._post_accumulate_grad_hooks for p in e.params):
            return self.model.log_prob_eager(x, ctx)           # a replay's backward is still due, or a hook must see the eager backward
        return _ReplayTrain.apply(e, x, ctx, *e.params)

    def _capture(self, x, ctx, params, frozen):
        # no garbage collection while the graphs are captured: a collected module tree may destroy CUDA graphs of its own, and those
        # calls invalidate a capture in progress (torch.cuda.graph collects once before it begins, not during)
        gc_was_enabled = gc.isenabled()
        gc.collect()
        gc.disable()
        try:
            with torch.cuda.device(x.device):
                return self._capture_on(x, ctx, params, frozen, x.device)
        finally:
            if gc_was_enabled:
                gc.enable()

    def _capture_on(self, x, ctx, params, frozen, device):
        from . import rng
        from .layers.flowlayer import live_capture
        e = _TrainEntry()
        e.device, e.params, e.frozen, e.generation, e.waiting = device, params, frozen, 0, None
        e.x = torch.empty(x.shape, device=device, dtype=x.dtype)
        e.ctx = None if ctx is None else torch.empty(ctx.shape, device=device, dtype=ctx.dtype)
        with torch.no_grad():
            e.x.copy_(x)
            if ctx is not None:
                e.ctx.copy_(ctx)
        # warm-up and capture draw random numbers: the generators are put back, so that the replay of this call draws what an eager call
        # would.  torch.autograd.grad leaves .grad alone.
        cpu_state, cuda_state = torch.get_rng_state(), torch.cuda.get_rng_state(device)
        cur = torch.cuda.current_stream(device)
        side = torch.cuda.Stream(device)
        side.wait_stream(cur)
        with _leaf_aliases(self.model, params) as leaves:
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    out = self.model.log_prob_eager(e.x, e.ctx)
                    torch.autograd.grad(out, leaves, torch.ones_like(out), allow_unused=True)
                del out
            cur.wait_stream(side)
            torch.cuda.synchronize(device)
            e.fwd, e.bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            del rng._capture_host_draws[:]
            with live_capture():
                with torch.cuda.graph(e.fwd, stream=side):
                    e.out = self.model.log_prob_eager(e.x, e.ctx)
                e.host_draws = list(rng._capture_host_draws)
                del rng._capture_host_draws[:]
                e.dlogp = torch.empty_like(e.out)
                # the forward's autograd graph is retained: the saved activations stay allocated between a forward and a backward replay
                with torch.cuda.graph(e.bwd, pool=e.fwd.pool(), stream=side):
                    grads = torch.autograd.grad(e.out, leaves, e.dlogp, retain_graph=True, allow_unused=True)
                    e.used = [g for g in grads if g is not None]
                    e.flat = _flatten_dense_tensors(e.used) if e.used else None
        e.slots = [i for i, g in enumerate(grads) if g is not None]
        e.used = [params[i] for i in e.slots]
        torch.set_rng_state(cpu_state); torch.cuda.set_rng_state(cuda_state, device)
        cur.wait_stream(side)
        e.versions = self._signature(frozen)
        return e


class GraphedTrainStep:
    """forward + loss + backward of a training step captured in ONE CUDA graph (torch.cuda.graph around the libcfpp launches, which go to
    torch's current stream): removes the host launch overhead of the 10^3 kernels of a specialist step.  A plain torch.optim.AdamW (what model.py:289
    builds) is not capturable and stays eager; contextflow_b200.optim.FusedAdamW is captured by attach_optimizer() and replayed by
    step().  Either way the optimizer reads the static .grad tensors the replay overwrites, so do NOT call zero_grad(set_to_none=True)
    between steps.  Inputs are copied into static buffers; shapes are fixed.
    `loss_fn(model, x, ctx, gt) -> scalar loss`."""

    def __init__(self, model, loss_fn, x, ctx, gt, warmup: int = 2):
        self.model, self.loss_fn = model, loss_fn
        self.static = (x.clone(), None if ctx is None else ctx.clone(), None if gt is None else gt.clone())
        params = [p for p in model.parameters() if p.requires_grad]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), eager_training():  # the model's own training graphs stay out of this step's warm-up
            for _ in range(warmup):                     # allocator warm-up, lazy initialisations (ActNorm flags, cached constants)
                for p in params:
                    p.grad = None
                loss_fn(model, *self.static).backward()
        torch.cuda.current_stream().wait_stream(side)
        for p in params:
            p.grad = None                                # the captured backward allocates the static .grad tensors in the graph's pool
        self.graph = torch.cuda.CUDAGraph()
        from . import rng
        from .layers.flowlayer import live_capture
        # live_capture: everything derived from a trainable parameter (log|det NN|, NN^-1, mixture tables, masked weights) is recomputed by
        # kernels recorded in the graph instead of being served from the version-keyed host caches the warm-up filled
        del rng._capture_host_draws[:]
        with live_capture(), torch.cuda.graph(self.graph):
            self.loss = loss_fn(model, *self.static)
            self.loss.backward()
        self.host_draws = list(rng._capture_host_draws)      # rng 'host' mode: device buffers that stand in for the CPU-generator draws
        del rng._capture_host_draws[:]

    def attach_optimizer(self, opt):
        """Capture `opt.step()` (contextflow_b200.optim.FusedAdamW: one multi-tensor kernel, step counter and bias corrections on the
        device) in a second graph over the static .grad tensors of the captured backward; `step()` then replays it.  Kept apart from the
        forward/backward graph so that a multi-GPU caller can all-reduce the gradients in between (sharded.GradAllReduce)."""
        from .optim import FusedAdamW
        if not isinstance(opt, FusedAdamW):
            raise TypeError('attach_optimizer needs a contextflow_b200.optim.FusedAdamW (a plain torch.optim.AdamW is not capturable)')
        plans = [opt._plan(gi, group) for gi, group in enumerate(opt.param_groups)]   # pointer tables and state buffers are built eagerly
        self.opt = opt
        self.opt_params = [p for plan in plans if plan is not None for p in plan['params']]
        self.opt_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.opt_graph):
            opt.step()
        return self

    def step(self):
        """Optimizer update from the gradients of the last replay (after an optional gradient all-reduce)."""
        self.opt.sync_learning_rate()
        self.opt_graph.replay()
        torch.autograd.graph.increment_version(self.opt_params)    # the replay wrote the parameters: invalidate what is cached on them

    def __call__(self, x, ctx, gt=None):
        self.static[0].copy_(x, non_blocking=True)
        if ctx is not None:
            self.static[1].copy_(ctx, non_blocking=True)
        if gt is not None:
            self.static[2].copy_(gt, non_blocking=True)
        for buf in self.host_draws:                            # same CPU-generator stream as an eager step (uniform.py:32)
            buf.copy_(torch.rand(buf.shape, dtype=buf.dtype))
        self.graph.replay()
        return self.loss
