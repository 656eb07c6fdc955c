"""Single-process, N-GPU `log_prob` (SURVEY §8e, "process model"): the reference's model.py / experiment_*.py are one process that
builds `torch.device('cuda:{gpu}')` and feeds un-sharded loaders (model.py:168-170,269-283), so the torchrun form (sharded.py) needs
caller code.  This form keeps the caller unchanged: the weights are replicated onto every visible device, a batch that arrives on the
model's device is cut into contiguous slices (sharded.shard_bounds), each slice is copied peer-to-peer to its device and scored there
by a replica (CUDA-graph replay per device, each on its own stream), and the (b_r, M) results are copied back and concatenated in batch
order on the caller's device.  No collective: per-sample log-likelihood shards trivially.

Turned on by FlowSequential.enable_multi_gpu() or CFPP_MULTI_GPU=1 (python -m contextflow_b200.run --multi-gpu ...); autograd calls and
small batches stay on the model's own device."""
from __future__ import annotations

import copy
import operator

import torch

from .sharded import shard_bounds

_version_of = operator.attrgetter('_version')


class ReplicatedLogProb:
    def __init__(self, model, devices=None, min_rows: int = 512):
        self.model = model
        self.min_rows = int(min_rows)
        self._devices = devices
        self._replicas = {}            # device index -> replica of the model
        self._sigs = {}                # device index -> source signature the replica was last refreshed at
        self._tensors = None
        self._all_initialized = False
        self._streams = {}

    # ---- replicas -------------------------------------------------------------------------------------------------------------
    def devices(self, primary):
        if self._devices is None:
            self._devices = [torch.device('cuda', i) for i in range(torch.cuda.device_count())]
        devs = [torch.device(d) for d in self._devices]
        return [primary] + [d for d in devs if d != primary]

    def _signature(self):
        ts = self._tensors
        if ts is None:
            ts = self._tensors = list(self.model.parameters()) + list(self.model.buffers())
        return hash(tuple(map(_version_of, ts))) ^ hash(tuple(t.data_ptr() for t in ts[:8]))

    def _replica(self, dev):
        r = self._replicas.get(dev.index)
        if r is None:
            r = copy.deepcopy(self.model)
            r.__dict__['_replicated'] = None           # a replica never fans out itself
            r.__dict__['_is_replica'] = True
            r = r.to(dev).eval()
            self._replicas[dev.index] = r
        return r

    def _sync(self, devs):
        """Replicas follow the source model: a replica's parameters / buffers are re-copied whenever a version counter moved (optimizer
        step, load_state_dict, ActNorm initialisation) since that replica was last refreshed.  Each replica keeps its own signature: a
        call that uses fewer devices than an earlier one leaves the others alone, and a later call on them must still refresh them."""
        sig = self._signature()
        reps, src = [], None
        for d in devs:
            fresh = d.index not in self._replicas          # a deepcopy made just now already holds the current values
            r = self._replica(d)
            if not fresh and self._sigs.get(d.index) != sig:
                if src is None:
                    src = list(self.model.parameters()) + list(self.model.buffers())
                with torch.no_grad():
                    for a, b in zip(list(r.parameters()) + list(r.buffers()), src):
                        a.copy_(b, non_blocking=True)
            self._sigs[d.index] = sig
            reps.append(r)
        return reps

    def _initialized(self):
        """ActNorm's data-dependent initialisation uses the statistics of the FIRST batch as a whole (actnorm.py:28-35): until every
        ActNorm has seen it, calls run on the model's own device."""
        if not self._all_initialized:
            flags = [b for n, b in self.model.named_buffers() if n.endswith('initialized')]
            self._all_initialized = all(int(f.item()) != 0 for f in flags)
        return self._all_initialized

    # ---- the call --------------------------------------------------------------------------------------------------------------
    def __call__(self, x, ctx=None):
        model = self.model
        B = x.shape[0]
        primary = x.device
        devs = self.devices(primary)
        n = min(len(devs), B // self.min_rows) if self.min_rows > 0 else len(devs)
        if n < 2 or not self._initialized():
            return model._log_prob_single(x, ctx)
        devs = devs[:n]
        # a peer copy moves one dense block: row slices of a contiguous batch are contiguous.  Made here, on the caller's stream before
        # `ready`, so that every slice's stream is ordered after it; the copies stay alive until the caller's stream has waited for all slices
        x = x.contiguous()
        ctx = None if ctx is None else ctx.contiguous()
        reps = self._sync(devs[1:])
        ready = torch.cuda.Event()
        cur = torch.cuda.current_stream(primary)
        ready.record(cur)                                           # x / ctx (and the replicas' refreshed weights) are complete at this point
        M = model.mixtures
        parts = []
        # Every device -- the caller's included -- works on its OWN non-blocking stream: it waits for `ready`, (pulls its slice from the
        # caller's device,) scores it and (pushes the (b, M) result into a buffer on the caller's device).  Two measured facts shape this
        # (tools/debug_mg2.py): torch's cross-device copy brackets the transfer with a two-way barrier between the current streams of both
        # devices, and a peer copy orders itself against the LEGACY DEFAULT stream of the device it touches -- which is torch's current
        # stream unless told otherwise -- so slices issued on the default streams ran one after the other.
        for r in range(n):
            lo, hi = shard_bounds(B, n, r)
            dev = devs[r]
            s = self._stream(dev)
            with torch.cuda.stream(s):
                s.wait_event(ready)
                if r == 0:
                    back = model._log_prob_single(x[lo:hi], None if ctx is None else ctx[lo:hi])
                else:
                    back = torch.empty((hi - lo, M), device=primary, dtype=torch.float32)
                    xs = torch.empty((hi - lo,) + tuple(x.shape[1:]), device=dev, dtype=x.dtype)
                    _peer_copy(xs, x[lo:hi], s)
                    cs = None
                    if ctx is not None:
                        cs = torch.empty((hi - lo,) + tuple(ctx.shape[1:]), device=dev, dtype=ctx.dtype)
                        _peer_copy(cs, ctx[lo:hi], s)
                    _peer_copy(back, reps[r - 1]._log_prob_single(xs, cs), s)
                done = torch.cuda.Event()
                done.record(s)
            parts.append((back, done))
        rows = []
        for back, done in parts:
            cur.wait_event(done)
            back.record_stream(cur)
            rows.append(back)
        return torch.cat(rows, 0)

    def _stream(self, dev):
        st = self._streams.get(dev.index)
        if st is None:
            st = self._streams[dev.index] = torch.cuda.Stream(dev)
        return st


def _peer_copy(dst, src, stream):
    """dst <- src (contiguous, same shape / dtype, possibly on different devices) on `stream` of the current device."""
    from . import _cabi
    assert dst.is_contiguous() and src.is_contiguous() and dst.numel() == src.numel() and dst.dtype == src.dtype
    rc = _cabi.lib().cfpp_copy_peer_async(_cabi.vp(dst.data_ptr()), dst.device.index, _cabi.vp(src.data_ptr()), src.device.index,
                                          dst.numel() * dst.element_size(), _cabi.vp(stream.cuda_stream))
    _cabi.check(rc, 'copy_peer_async')
