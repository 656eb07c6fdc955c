"""Generate tests/golden/extras.npz by executing the UNMODIFIED reference classes that create_model never builds but that can be
constructed directly: the standalone Sigmoid / Softplus flow layers (layers/activations.py:228-264) and StudentMixtureDistribution
(layers/distributions/student.py:44-111).
    CFPP_REFERENCE=<upstream checkout>/contextflow python tests/golden/make_golden_extras.py"""
import os, sys
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from contextflow_b200 import synth  # noqa: E402
from tests.golden.make_golden import import_reference  # noqa: E402

STUDENT = dict(size=(4, 3, 2), mixtures=3, B=5)


def main():
    import_reference()
    from layers.activations import Sigmoid, Softplus
    from layers.distributions.student import StudentMixtureDistribution
    tape = synth.NoiseTape('extras')
    rec = {}
    x = (tape.randn((7, 19)) * 3.0).float()
    x[0, 0], x[0, 1], x[1, 0] = 25.0, -25.0, 0.0                       # softplus threshold branch on both sides
    rec['act_x'] = x.numpy()
    for T in (1.0, 2.5):
        lay = Sigmoid(temperature=T, eps=1e-6)
        z, ldj = lay(x)
        rec[f'sig_z_{T}'], rec[f'sig_ldj_{T}'] = z.numpy(), ldj.numpy()
        rec[f'sig_rev_{T}'] = lay.reverse(z).numpy()
    lay = Softplus()
    z, ldj = lay(x)
    rec['sp_z'], rec['sp_ldj'], rec['sp_rev'] = z.numpy(), ldj.numpy(), lay.reverse(z).numpy()
    xg = x.clone().requires_grad_(True)                                   # gradients of sum(z * a) + sum(ldj * b)
    a, b = tape.randn((7, 19)).float(), tape.randn((7,)).float()
    rec['act_a'], rec['act_b'] = a.numpy(), b.numpy()
    z, ldj = Sigmoid(temperature=2.5)(xg); ((z * a).sum() + (ldj * b).sum()).backward(); rec['sig_dx_2.5'] = xg.grad.numpy().copy(); xg.grad = None
    z, ldj = Softplus()(xg); ((z * a).sum() + (ldj * b).sum()).backward(); rec['sp_dx'] = xg.grad.numpy().copy()
    torch.manual_seed(0)
    D, H, W = STUDENT['size']
    dist = StudentMixtureDistribution(STUDENT['size'], mixtures=STUDENT['mixtures'])
    sd = dist.state_dict(); synth.fill_state(sd, 'student'); dist.load_state_dict(sd)
    xs = (tape.randn((STUDENT['B'], D, H, W)) * 1.5).float()
    rec['stu_x'] = xs.numpy()
    with torch.no_grad():
        rec['stu_logp'] = dist.log_prob(xs).numpy()
        rec['stu_logp64'] = dist.double().log_prob(xs.double()).numpy()
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', 'extras.npz'), **rec)
    print('extras:', {k: v.shape for k, v in rec.items()})


if __name__ == '__main__':
    main()
