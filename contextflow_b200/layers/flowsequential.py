"""Flow containers (reference layers/flowsequential.py): FlowSequential.forward/log_prob (:18-30) accumulates the per-layer
ldj into a (B, M) log-det and adds the base log-prob; FlowInvSequential.sample (:60-69) drives the encoder flows."""
import torch
import torch.nn as nn

from .. import ops, training

__all__ = ['FlowSequential', 'FlowInvSequential']


class FlowSequential(nn.Module):
    def __init__(self, dist, *modules):
        super().__init__()
        self.dist = dist
        self.mixtures = dist.M
        for i, module in enumerate(modules):
            self.add_module(str(i), module)
        self.sequence_modules = modules
        from .splitprior import SplitPrior
        from .squeeze import Squeeze
        for m, nxt in zip(modules, modules[1:]):                 # SplitPrior -> Squeeze (model.py:153-158, 125-127): the kept half is handed over
            if isinstance(m, SplitPrior) and isinstance(nxt, Squeeze) and tuple(getattr(nxt, 'p', getattr(nxt, 'factor', (0, 0)))) == (2, 2):
                m._view_ok = True                                # as a view; the squeeze kernel reads it through the batch stride (no copy)
        import os
        self._graphed = None
        self._graphed_train = None
        scoring, training_ = os.environ.get('CFPP_CUDA_GRAPHS', '0') == '1', os.environ.get('CFPP_CUDA_GRAPHS_TRAIN', '0') == '1'
        if scoring or training_:
            self.enable_cuda_graphs(scoring, training=training_)

    def __iter__(self):
        yield from self.sequence_modules

    def __deepcopy__(self, memo):
        """copy.deepcopy(model) (EMA / best-model snapshots): the execution plan, encoder batches and captured graphs hold ctypes
        descriptors and device pointers of THIS module tree, so the copy starts without them and rebuilds them lazily."""
        import copy
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ('_fastpath', '_graphed', '_graphed_train', '_groups', '_replicated'):
                continue
            new.__dict__[k] = copy.deepcopy(v, memo)
        new.__dict__['_groups'] = None
        new.__dict__['_graphed'] = None
        new.__dict__['_graphed_train'] = None
        training_ = self.__dict__.get('_graphed_train') is not None
        if self._graphed is not None or training_:
            new.enable_cuda_graphs(self._graphed is not None, training=training_)
        return new

    def _apply(self, fn, *args, **kwargs):
        """.to() / .cuda() / .double(): parameters may be re-created, so captured graphs and their cached tensor list are dropped."""
        out = super()._apply(fn, *args, **kwargs)
        for name in ('_graphed', '_graphed_train'):
            g = self.__dict__.get(name)
            if g is not None:
                g.invalidate()
        return out

    def _encoder_groups(self):
        """{index of first member layer: EncoderBatch}: runs of layers whose context encoders can share one launch.  A run
        ends at any layer that draws noise itself (Augment, Dequantization) or whose context_net is an opaque callable."""
        if getattr(self, '_groups', None) is not None:
            return self._groups
        from ._encoder_desc import EncoderBatch
        from .augment import Augment
        from .dequantize import Dequantization
        groups, cur, start = {}, [], None

        def close():
            nonlocal cur, start
            if len(cur) > 1:
                groups[start] = EncoderBatch(cur)
            cur, start = [], None

        for i, m in enumerate(self.sequence_modules):
            if isinstance(m, (Augment, Dequantization)):
                close(); continue
            owner = m.dist if hasattr(m, 'dist') and hasattr(m.dist, '_plan') else m
            net = getattr(owner, 'context_net', None)
            if net is None or not hasattr(owner, '_plan'):
                continue
            fused = owner._plan.fused_for(net)
            if fused is None:
                close(); continue
            if EncoderBatch.is_lookup(fused):
                continue
            if start is None:
                start = i
            cur.append((owner._plan, fused))
        close()
        self._groups = groups
        return groups

    def forward(self, input, context=None):
        B = input.shape[0]
        out = input
        terms = []
        if torch.is_grad_enabled():
            ops.begin_training_step()                               # per-step caches of the backward pass (context sort of embed_scatter) start empty
        # under autograd every layer evaluates its own encoder (trainable encoders run their module tree: training.encode), in layer order
        groups = self._encoder_groups() if (context is not None and not torch.is_grad_enabled()) else {}
        for i, module in enumerate(self.sequence_modules):
            batch = groups.get(i)
            if batch is not None and batch.ready():
                batch.run(context)
            out, ldj = module(out, context)
            terms.append(ldj)                                   # (B,), (B,1) broadcast or (B,M)   (flowsequential.py:23)
        logprob = self.dist.log_prob(out, context)
        if training.wants_grad(logprob, *terms):
            return out, training.LdjSumFn.apply(logprob, self.mixtures, *terms)
        # logdet = ((0 + ldj_0) + ldj_1) + ...; logprob + logdet  (flowsequential.py:20-27), same order, one launch
        return out, ops.ldj_sum(terms, B, self.mixtures, input.device, last=logprob)

    def enable_cuda_graphs(self, flag: bool = True, training: bool = False):
        """flag: replay `log_prob` from a captured CUDA graph (one graph per input shape) whenever autograd is off: removes the
        per-launch host overhead of the ~10^2 kernels of a forward.
        training: also replay `log_prob` under autograd, from a forward and a backward graph per input shape (graphed.GraphedTrainLogProb),
        for a training loop that keeps its own loss, backward() and optimizer step; the ~10^3 launches of a training step then become
        two graph launches.  The first call at a new shape, and the first after a load_state_dict, run eagerly; the second captures.
        Calls with an input that requires grad, with a gradient hook on a parameter, inside another capture or under a replayed noise
        tape stay eager.
        Both off by default; `python -m contextflow_b200.run` turns them on with CFPP_CUDA_GRAPHS=1 and CFPP_CUDA_GRAPHS_TRAIN=1.
        forward() (which also returns z) always runs eagerly."""
        from ..graphed import GraphedLogProb, GraphedTrainLogProb
        self._graphed = GraphedLogProb(self) if flag else None
        self._graphed_train = GraphedTrainLogProb(self) if training else None
        return self

    def log_prob_eager(self, input, context=None):
        """log_prob launched kernel by kernel: the fused plan (layers/_fastpath.py) when it applies, else layer by layer."""
        import os
        if os.environ.get('CFPP_FASTPATH', '1') != '0':
            fp = getattr(self, '_fastpath', None)
            if fp is None:
                from ._fastpath import FastLogProb
                fp = FastLogProb(self)
                object.__setattr__(self, '_fastpath', fp)
            if fp.usable(input, context):
                return fp(input, context)
        return self.forward(input, context)[1]

    def enable_multi_gpu(self, flag: bool = True, devices=None, min_rows: int = 512):
        """Single-process N-GPU log_prob (SURVEY §8e process model, contextflow_b200/multigpu.py): batches of at least 2 * min_rows rows that
        arrive on the model's device under no_grad are cut into contiguous slices, scored by weight replicas on every visible device and
        concatenated back in order on the caller's device.  Also turned on by CFPP_MULTI_GPU=1."""
        from ..multigpu import ReplicatedLogProb
        object.__setattr__(self, '_replicated', ReplicatedLogProb(self, devices, min_rows) if flag else None)
        return self

    def log_prob(self, input, context=None):
        rep = self.__dict__.get('_replicated', False)
        if rep is False:                                         # first call: the environment decides (a replica carries None)
            import os
            rep = None
            if os.environ.get('CFPP_MULTI_GPU', '0') == '1' and not self.__dict__.get('_is_replica'):
                self.enable_multi_gpu()
                rep = self.__dict__['_replicated']
            else:
                object.__setattr__(self, '_replicated', None)
        if (rep is not None and input.is_cuda and not torch.is_grad_enabled() and not torch.cuda.is_current_stream_capturing()
                and torch.cuda.device_count() > 1):
            from .. import rng
            if rng._source is None and rng._recorder is None:
                return rep(input, context)
        return self._log_prob_single(input, context)

    def _log_prob_single(self, input, context=None):
        if torch.is_grad_enabled():
            ops.begin_training_step()
            gt = self.__dict__.get('_graphed_train')
            if gt is not None and input.is_cuda:
                return gt(input, context)
        g = getattr(self, '_graphed', None)
        if g is not None and input.is_cuda and not torch.is_grad_enabled() and not torch.cuda.is_current_stream_capturing():
            from .. import rng
            if rng._source is None and rng._recorder is None:  # replayed noise tapes / draw recording (tests) are host-driven: stay eager
                return g(input, context)
        return self.log_prob_eager(input, context)

    def reverse(self, z, context=None):
        """The layer loop of flowsequential.py:34-37 from a given latent z (what `sample` runs after drawing z).  The image
        prologue's four reverses + Augment.reverse run as one kernel when the stack starts the way create_model builds it."""
        mods = list(self.sequence_modules)
        tail = self._prologue_tail()
        out = z
        for module in reversed(mods[tail:] if tail else mods):
            out = module.reverse(out, context)
        if tail:
            n0, n1 = mods[1], mods[2]
            s0, t0, _ = n0.host_constants(); s1, t1, _ = n1.host_constants()
            aug = mods[4].aug_size if tail == 5 else 0
            out = ops.prologue_inv(out, out.shape[1] - aug, s1, t1, s0, t0, do_floor=True)
        return out

    def _prologue_tail(self):
        """Number of leading layers covered by the fused inverse prologue (0, 4 or 5): Dequantization, Normalization x2 (scalar),
        LogitTransform [, Augment on channels] -- model.py:97-100,121-123."""
        import os
        from .augment import Augment
        from .dequantize import Dequantization
        from .normalize import Normalization
        from .transforms import LogitTransform
        mods = list(self.sequence_modules)
        if os.environ.get('CFPP_FASTPATH', '1') == '0' or len(mods) < 4:
            return 0
        if not (isinstance(mods[0], Dequantization) and isinstance(mods[1], Normalization) and isinstance(mods[2], Normalization)
                and isinstance(mods[3], LogitTransform) and mods[1].scale.numel() == 1 and mods[2].scale.numel() == 1):
            return 0
        if len(mods) > 4 and isinstance(mods[4], Augment) and mods[4].split_dim == 1:
            return 5
        return 4

    def sample(self, n_samples, context=None):
        """flowsequential.py:32-39: z ~ dist, then every layer's reverse from last to first."""
        z, _ = self.dist.sample(n_samples, context)
        return self.reverse(z, context)


class FlowInvSequential(nn.Module):
    def __init__(self, dist, *modules):
        super().__init__()
        self.dist = dist
        for i, module in enumerate(modules):
            self.add_module(str(i), module)
        self.sequence_modules = modules

    def __iter__(self):
        yield from self.sequence_modules

    def forward(self, input, context=None):
        return self.sample(input, context)

    def log_prob(self, input, context=None):
        raise RuntimeError('InverseFlow does not support log_prob, see Flow instead.')

    def sample(self, input, context=None):
        out, logprob = self.dist.sample(input.size(0), context)
        for module in self.sequence_modules:
            out, ldj = module(out, context)
            logprob = logprob - (ldj if ldj.dim() == logprob.dim() else ldj.squeeze(-1))
        return out, logprob
