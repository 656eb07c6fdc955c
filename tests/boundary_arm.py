"""One arm of the end-to-end boundary test (run as a subprocess by tests/test_gpu_boundary.py):

    python tests/boundary_arm.py <replacement|reference> <ad|cl> <out.json>

Drives the reference's UNMODIFIED `AdExperiment` / `ClExperiment` (experiment_ad.py / experiment_cl.py) -- eval_epoch, train_epoch,
save(), load() of a generalist checkpoint into a specialist (experiment_ad.py:304-323) -- over either this repo's layers
(`replacement`: contextflow_b200.run.install_layers + the fused AdamW + CUDA graphs for inference, exactly what `python -m contextflow_b200.run
model.py` sets up) or the reference's own torch layers (`reference`, TF32 off) on the same GPU, with identical weights
(synth.fill_state), identical in-memory loaders and identical generator seeds.  With CFPP_RNG=reference both arms consume
torch's generators identically, so every number they print must agree within the fp32 parity gates."""
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))


def main(arm, kind, out_path):
    if arm == 'replacement':
        os.environ.setdefault('CFPP_CUDA_GRAPHS', '1')          # what run.py sets
        os.environ['CFPP_RNG'] = 'reference'
    import torch
    import torch.nn as nn
    import torch.optim as optim
    from torch.optim.lr_scheduler import StepLR
    import refshim
    M = refshim.import_reference(replacement=(arm == 'replacement'))
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    from contextflow_b200 import synth
    if arm == 'replacement':
        import contextflow_b200.layers as L
        assert M.FlowSequential is L.FlowSequential, 'model.py did not pick up the replacement layers'
        if os.environ.get('CFPP_FUSED_ADAMW', '1') != '0':      # what run.py installs: optim.AdamW (model.py:289) builds the fused optimizer
            from contextflow_b200 import optim as _optim
            _optim.install()
    dev = torch.device(os.environ.get('CFPP_BND_DEVICE', 'cuda:0'))
    if kind == 'ad':
        from experiment_ad import AdExperiment as Exp
        gen = synth.variant('cfg4', num_blocks=1, block_size=2)
        spec = synth.variant('cfg4', num_blocks=1, block_size=2, generalist=False, contextflow=True, enc_emb='onehot', enc_type='uniform')
        mixtures, weight = 1, None
        B, nb = 96, 3
    else:
        from experiment_cl import ClExperiment as Exp
        gen = synth.variant('cfg2', num_blocks=2, block_size=1, generalist=True, contextflow=False)
        spec = synth.variant('cfg2', num_blocks=2, block_size=1)      # onehot + vardeq, --contextflow (BASELINE cfg2's encoder)
        mixtures, weight = 10, torch.ones(10)
        B, nb = 48, 3

    def loader(conf, tag, sizes):
        out = []
        for i, b in enumerate(sizes):
            x, c = synth.make_inputs(conf, b, f'{tag}{i}')
            gt = (synth.uniform(f'{tag}gt{i}', (b,)) * mixtures).long().clamp_(0, mixtures - 1)
            out.append((x, gt, c))
        return out

    def experiment(conf, path, generalist):
        torch.manual_seed(0)
        net = refshim.create_model(M, conf)
        sd = net.state_dict(); synth.fill_state(sd, 'bnd'); net.load_state_dict(sd)
        net = net.to(dev)
        opt = optim.AdamW(filter(lambda p: p.requires_grad, net.parameters()), lr=1e-3)          # model.py:289-290
        sch = StepLR(opt, step_size=2, gamma=0.1)
        crit = None if weight is None else nn.CrossEntropyLoss(weight=weight.to(dev))
        tr = loader(conf, 'tr', [B] * nb); va = loader(conf, 'va', [B, B, B // 2 + 1])            # ragged last batch
        cfg = dict(epochs=2, device=dev, dataset=conf['cfg']['dataset'], name='bnd', checkpoint_path=path, save_checkpoint=True, wandb=False,
                   verbose=False, eval_epochs=1, log_interval=float('inf'), lr=1e-3, grad_clip_norm=None, generalist=generalist)
        return Exp(conf['data_size'], net, tr, va, va, opt, crit, sch, **cfg), net, va

    def evaluate(exp, va, seed):
        torch.manual_seed(seed)
        r = exp.eval_epoch(va, 1)
        loss, scores = float(r[0]), [float(v) for v in r[-1]][:256]
        extra = float(r[1]) if kind == 'cl' else None
        return dict(loss=loss, scores=scores, log_px=extra)

    res = {}
    tmp = tempfile.mkdtemp()
    gpath = os.path.join(tmp, 'bnd_generalist.pt')                 # 'generalist' in the path selects the strict=False branch of load()
    exp, net, va = experiment(gen, gpath, True)
    res['gen_eval0'] = evaluate(exp, va, 1)
    torch.manual_seed(2)
    res['gen_train'] = float(exp.train_epoch(5))                   # epoch > warmup_epochs: lr as configured
    res['gen_eval1'] = evaluate(exp, va, 3)
    exp.save()
    # specialist: load the generalist checkpoint (missing keys = the context networks), evaluate, train, evaluate
    sexp, snet, sva = experiment(spec, os.path.join(tmp, 'bnd_specialist.pt'), False)
    import io, contextlib
    buf = io.StringIO()
    _tl = torch.load
    torch.load = lambda p, **kw: _tl(p, weights_only=False, **kw)   # the checkpoint holds the config dict (torch >= 2.6 defaults to weights_only)
    with contextlib.redirect_stdout(buf):
        sexp.load(gpath)
    torch.load = _tl
    res['spec_trainable'] = sorted(k for k, p in snet.named_parameters() if p.requires_grad)
    res['spec_eval0'] = evaluate(sexp, sva, 4)
    torch.manual_seed(5)
    res['spec_train'] = float(sexp.train_epoch(5))
    res['spec_eval1'] = evaluate(sexp, sva, 6)
    res['param_abs_sum'] = float(sum(p.detach().double().abs().sum() for p in snet.parameters()))
    if arm == 'replacement':
        from contextflow_b200 import _cabi
        res['launches'] = _cabi.launch_count()
        res['graphs'] = len(snet._graphed._entries) if getattr(snet, '_graphed', None) is not None else 0
    json.dump(res, open(out_path, 'w'))


if __name__ == '__main__':
    main(*sys.argv[1:4])
