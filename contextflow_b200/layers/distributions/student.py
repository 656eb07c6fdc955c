"""StudentMixtureDistribution (reference layers/distributions/student.py:44-111, `--dist tdist`).  create_model cannot build it
(model.py:163 passes `components=`, which student.py:44 rejects), but the class can be constructed directly.  log_prob runs CUDA kernels:
for scoring, and under autograd (training.StudentMixtureFn) with gradients for mG, sG, wG, mS, sS, wS and for the input, so the prior
trains as FlowSequential.dist or inside a SplitPrior.  vS stays frozen, as in the reference (student.py:59)."""
import torch
import torch.nn as nn

from ... import ops, training
from ..flowlayer import PackCache, inference_only

__all__ = ['StudentMixtureDistribution']


class StudentMixtureDistribution(nn.Module):
    """Sum of a K = 8 Gaussian-mixture log-density and a K = 8 Student-t mixture log-density per mixture m (student.py:95-98); the
    reference sets context_net = None and contextflow = False whatever is passed (student.py:64-65)."""

    def __init__(self, size, mixtures=2, context_net=None, contextflow=False):
        super().__init__()
        self.size = size
        D, H, W = size
        self.M, self.K = mixtures, 8
        M, K = self.M, self.K
        self.mG = nn.Parameter(torch.randn(M, K, D, H, W))
        self.sG = nn.Parameter(torch.ones(M, K, D, H, W))
        self.wG = nn.Parameter(torch.randn(M, K))
        self.mS = nn.Parameter(torch.randn(M, K, D, H, W))
        self.sS = nn.Parameter(torch.ones(M, K, D, H, W))
        self.wS = nn.Parameter(torch.randn(M, K))
        v_init = torch.linspace(1, 10, K).view(1, K, 1, 1, 1)
        self.vS = nn.Parameter(v_init.repeat(M, 1, D, H, W))
        self.vS.requires_grad_(False)
        self.context_net = None
        self.contextflow = False
        self._tables = PackCache()

    def forward(self, input, context=None):
        return self.log_prob(input, context)

    def log_prob(self, input, context=None):
        if training.wants_grad(input, self.mG, self.sG, self.wG, self.mS, self.sS, self.wS):
            inference_only(self.vS)
            return training.StudentMixtureFn.apply(input, self, 0, self.mG, self.sG, self.wG, self.mS, self.sS, self.wS)
        src = [self.mG, self.sG, self.wG, self.mS, self.sS, self.wS, self.vS]
        for p in src:
            inference_only(p)
        inference_only(input)
        table = self._tables.get('student', src, lambda: ops.student_table(*[p.detach() for p in src]))
        return ops.student_logprob(input, table, self.M, self.K)
