"""SplitPrior: factor out the second half of the channels under a (context-conditioned) mixture prior
(reference layers/splitprior.py:7-15)."""
from .. import ops, training
from .flowlayer import FlowLayer, inference_only


class SplitPrior(FlowLayer):
    def __init__(self, dist):
        super().__init__()
        self.dist = dist

    def forward(self, x, context=None):
        d = self.dist
        if hasattr(d, 'mS') and training.wants_grad(x, d.mG, d.sG, d.wG, d.mS, d.sS, d.wS):     # Student-t mixture: it has an mG too
            inference_only(d.vS)                                    # the degrees of freedom have no backward kernel (frozen in the reference)
            return training.StudentMixtureFn.apply(x, d, x.shape[1] // 2, d.mG, d.sG, d.wG, d.mS, d.sS, d.wS)
        if not getattr(d, 'context_net', None) and hasattr(d, 'mG') and training.wants_grad(x, d.mG, d.sG, d.wG):
            return training.SplitPriorFn.apply(x, d.mG, d.sG, d.wG, d)
        if getattr(d, 'context_net', None) and hasattr(d, 'mG') and training.wants_grad(x, *d.context_net.parameters()):
            tables = training._lookup_tables(d)
            if tables is None:
                raise NotImplementedError('training a split prior whose context_net is not the embed + eyesample lookup has no backward '
                                          'kernel yet')
            ctx2 = context[0] if isinstance(context, list) else context
            return training.GmmCtxFn.apply(x, ctx2, d, x.shape[1] // 2, d.mG, d.sG, d.wG, *tables)
        half = x.shape[1] // 2
        ldj = self.dist.log_prob(x[:, half:], context)         # read in place through the batch stride, (B, M)
        if getattr(self, '_view_ok', False) and x.is_contiguous() and x.shape[3] % 8 == 0 and (half * x.shape[2] * x.shape[3]) % 4 == 0:
            return x[:, :half], ldj                             # the next layer is a 2x2 Squeeze that reads this view in place (ops.squeeze)
        return ops.slice_channels(x, 0, half), ldj

    def reverse(self, z, context=None):
        # splitprior.py:17-21 calls self.dist.sample(self.C, context) but SplitPrior never defines `C`: the reference raises
        # AttributeError here, so models with split priors (cfg2, cfg3) have no executable inverse to be on par with
        raise AttributeError("'SplitPrior' object has no attribute 'C'")

    def logdet(self, input, context=None):
        return self.forward(input, context)[1]
