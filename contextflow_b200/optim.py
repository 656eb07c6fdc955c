"""Fused AdamW: torch.optim.AdamW (what the reference builds, model.py:289) with `step()` as ONE multi-tensor kernel whose step counter
and bias corrections live on the device, so the update can sit inside the training step's CUDA graph (GraphedTrainStep).  It subclasses
torch.optim.AdamW: param_groups, StepLR (model.py:290), state_dict / load_state_dict (experiment_ad.py:298,319) behave as before; the
state per parameter is torch's ({'step', 'exp_avg', 'exp_avg_sq'}).  `install()` makes `torch.optim.AdamW` name this class, which is
how `python -m contextflow_b200.run model.py` gives the unchanged model.py the fused optimizer."""
from __future__ import annotations

import numpy as np
import torch

from . import _cabi

_TorchAdamW = torch.optim.AdamW


class FusedAdamW(_TorchAdamW):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False, **kw):
        if amsgrad or kw.get('maximize'):
            raise NotImplementedError('FusedAdamW covers the configuration the reference uses (model.py:289): amsgrad=False, maximize=False')
        for k in ('foreach', 'fused', 'capturable', 'differentiable', 'maximize'):
            kw.pop(k, None)
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False)
        self._plans = {}

    # one plan per param group: pointer / chunk tables on the device, the step state and the learning rate as device scalars
    def _plan(self, gi, group):
        ps = [p for p in group['params'] if p.grad is not None]
        for p in ps:
            if not p.is_cuda or p.dtype != torch.float32 or p.grad.dtype != torch.float32 or not p.is_contiguous() or not p.grad.is_contiguous():
                raise RuntimeError('FusedAdamW updates contiguous float32 CUDA parameters only (no CPU fallback)')
            st = self.state[p]
            if len(st) == 0:
                st['step'] = torch.zeros((), dtype=torch.float32, device=p.device)
                st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
        key = tuple((p.data_ptr(), p.grad.data_ptr(), self.state[p]['exp_avg'].data_ptr()) for p in ps)
        plan = self._plans.get(gi)
        if plan is not None and plan['key'] == key:
            return plan
        if not ps:
            return None
        dev = ps[0].device
        chunk = int(_cabi.lib().cfpp_adamw_chunk())
        ptrs = np.array([[p.data_ptr(), p.grad.data_ptr(), self.state[p]['exp_avg'].data_ptr(), self.state[p]['exp_avg_sq'].data_ptr()] for p in ps],
                        dtype=np.uint64).reshape(-1)
        chunks = []
        for t, p in enumerate(ps):
            n = p.numel()
            for first in range(0, n, chunk):
                chunks.append((t, first, min(chunk, n - first)))
        old = plan['state'] if plan is not None else None
        state = old if old is not None else torch.zeros(3, dtype=torch.float32, device=dev)
        if old is None:                                   # resume (load_state_dict): the per-parameter step counters are all equal
            state[0] = float(self.state[ps[0]]['step'])
        plan = dict(key=key, params=ps, n_chunks=len(chunks), state=state,
                    tensors=torch.from_numpy(ptrs.view(np.int64)).to(dev), chunks=torch.tensor(chunks, dtype=torch.int32, device=dev).reshape(-1),
                    lr=torch.full((1,), float(group['lr']), dtype=torch.float32, device=dev), lr_host=float(group['lr']))
        self._plans[gi] = plan
        return plan

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        capturing = torch.cuda.is_current_stream_capturing()
        for gi, group in enumerate(self.param_groups):
            plan = self._plan(gi, group)
            if plan is None:
                continue
            if plan['lr_host'] != float(group['lr']) and not capturing:        # a scheduler moved the learning rate (model.py:290)
                plan['lr'].fill_(float(group['lr'])); plan['lr_host'] = float(group['lr'])
            b1, b2 = group['betas']
            dev = plan['state'].device
            with torch.cuda.device(dev):
                rc = _cabi.lib().cfpp_adamw_step(_cabi.vp(plan['tensors'].data_ptr()), _cabi.vp(plan['chunks'].data_ptr()), plan['n_chunks'],
                                                 _cabi.vp(plan['state'].data_ptr()), _cabi.vp(plan['lr'].data_ptr()), float(b1), float(b2),
                                                 float(group['eps']), float(group['weight_decay']), _cabi.vp(torch.cuda.current_stream(dev).cuda_stream))
            _cabi.check(rc, 'adamw_step')
            if not capturing:
                # the kernel writes through raw pointers: bump the version counters so that every value cached on them (log|det NN|,
                # NN^-1, mixture tables, packed weights, captured log_prob graphs, multi-GPU replicas) is rebuilt
                torch.autograd.graph.increment_version(plan['params'])
        return loss

    def sync_learning_rate(self):
        """Push the host learning rates (a scheduler may have changed them) to the device scalars a captured step reads."""
        for gi, group in enumerate(self.param_groups):
            plan = self._plans.get(gi)
            if plan is not None and plan['lr_host'] != float(group['lr']):
                plan['lr'].fill_(float(group['lr'])); plan['lr_host'] = float(group['lr'])

    def state_dict(self):
        for plan in self._plans.values():                    # torch keeps a step counter per parameter: mirror the group's device counter into them
            for p in plan['params']:
                self.state[p]['step'].copy_(plan['state'][0])
        return super().state_dict()

    def load_state_dict(self, sd):
        super().load_state_dict(sd)
        self._plans = {}


def install():
    """torch.optim.AdamW -> FusedAdamW for code that is about to be imported (the reference's model.py does `import torch.optim as optim`)."""
    torch.optim.AdamW = FusedAdamW
    return FusedAdamW
