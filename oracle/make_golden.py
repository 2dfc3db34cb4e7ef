"""Generates tests/golden/* by running the UNMODIFIED reference (a checkout of eladhoffer/convNet.pytorch, named by
the environment variable B200_REFERENCE).  Run from the repo root:  B200_REFERENCE=<checkout> python oracle/make_golden.py
The fixtures pin (a) the oracle restatement (oracle/ref_model.py), (b) the re-authored host code
(models, regimes, trainer) and (c) -- through the GPU tests -- the CUDA pipeline.
The reference is not needed at test time: tests read only the committed fixtures, in the encodings of
oracle/fixtures.py.
"""
import json
import os
import sys
from copy import deepcopy

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle.fixtures import bf16_bits, synth_record, synthetic_momentum  # noqa: E402

REF = os.environ.get('B200_REFERENCE')
OUT = os.path.join(ROOT, 'tests', 'golden')


def import_reference():
    if not REF:
        raise SystemExit('make_golden.py: set B200_REFERENCE to a checkout of the reference')
    sys.path.insert(0, REF)
    import models as ref_models            # noqa: E402
    import trainer as ref_trainer          # noqa: E402
    from utils import optim as ref_optim   # noqa: E402
    from utils import cross_entropy as ref_ce  # noqa: E402
    return ref_models, ref_trainer, ref_optim, ref_ce


def tensor_stats(sd):
    out = {}
    for k, v in sd.items():
        v = v.double().flatten()
        out[k] = {'shape': list(sd[k].shape), 'sum': float(v.sum()), 'abs': float(v.abs().sum()),
                  'head': [float(t) for t in v[:4]]}
    return out


SAMPLE = 256   # elements per tensor kept of gradients and updated parameters


def sample_index(numel, rng):
    return np.arange(numel) if numel <= SAMPLE else np.sort(rng.choice(numel, SAMPLE, replace=False))


def mobilenet_v2_fixture(ref_models, ref_trainer, ref_optim, ref_ce):
    """MobileNet-v2 (config C4's family) through the reference Trainer on 16 x 3x96x96 inputs, default init (seed 123),
    classifier dropout ACTIVE (generator re-seeded before every step so that a restatement draws the same masks):
    step 1 is recorded in full (logits, loss, gradient norms + heads, post-step parameter statistics), step 2 by its
    loss.  Default-init MobileNet-v2 is ill-conditioned (fp32 vs fp64 gradients of the SAME code differ by 3e-3..1e-2,
    measured with the restatement), so only step 1 supports tight bounds.  The model itself is re-created from the
    seed (test_model_factories_match_reference_init pins that)."""
    torch.manual_seed(123)
    model = ref_models.mobilenet_v2(dataset='imagenet')
    x, y, rec = synth_record(16, (3, 96, 96), 1000)
    opt = ref_optim.OptimRegime(model, model.regime)
    tr = ref_trainer.Trainer(model, ref_ce.CrossEntropyLoss(), opt, device_ids=None, device='cpu',
                             dtype=torch.float, print_freq=1000)
    model.train()
    opt.zero_grad(); opt.update(0, 0)
    wd_names = [n for n, _ in opt.regularizer.regularization_list[0]._named_parameters]
    torch.manual_seed(1000)
    out = model(x); loss = tr.criterion(out, y); loss.backward()
    gn = {n: float(p.grad.norm()) for n, p in model.named_parameters()}
    gh = {n: p.grad.flatten()[:4].clone().numpy() for n, p in model.named_parameters()}
    opt.step()
    tr.training_steps += 1
    post = tensor_stats(model.state_dict())
    torch.manual_seed(1001)
    _, loss2, _ = tr._step(x, y, training=True)
    np.savez(os.path.join(OUT, 'mobilenet_v2_summary.npz'), **rec, logits=out.detach().numpy(),
             loss=np.float64(float(loss)), loss_step2=np.float64(float(loss2)), grad_names=np.array(list(gn.keys())),
             grad_norms=np.array(list(gn.values())), grad_heads=np.stack([gh[n] for n in gn]),
             wd_names=np.array(wd_names), post_names=np.array(list(post.keys())),
             post_sums=np.array([post[k]['sum'] for k in post]), post_abs=np.array([post[k]['abs'] for k in post]))
    print('mobilenet_v2 fixture written')


NEIGHBOURS = [('resnext50', 'resnext', dict(dataset='imagenet', depth=50)),
              ('resnet_se50', 'resnet_se', dict(dataset='imagenet', depth=50)),
              ('resnext_se50', 'resnext_se', dict(dataset='imagenet', depth=50)),
              ('mobilenet_v1', 'mobilenet', dict(dataset='imagenet')),
              # the hot-path families themselves, in double precision (their fp32 fixtures above carry rounding noise)
              ('resnet50', 'resnet', dict(dataset='imagenet', depth=50)),
              ('resnet18', 'resnet', dict(dataset='imagenet', depth=18)),
              ('mobilenet_v2', 'mobilenet_v2', dict(dataset='imagenet'))]


def neighbours_fixture(ref_models, ref_ce):
    """Grouped convolutions (ResNeXt), squeeze-excitation gates (resnet_se / resnext_se: one SEBlock shared by the
    blocks of a stage) and MobileNet-v1 (depthwise with bias): one training-mode forward/backward of the UNMODIFIED
    reference models on 8 x 3x96x96 inputs at default init (seed 123), run in DOUBLE precision (the fp32 runs of these
    networks carry 1e-3 of rounding noise in the SE variants) -- logits, loss, every parameter-gradient norm,
    running-statistics sums.  Pins oracle.ref_model's restatement of those families (tests/test_oracle_golden.py)."""
    blob = {}
    x, y, rec = synth_record(8, (3, 96, 96), 1000, seed=7)
    blob.update(rec)
    crit = ref_ce.CrossEntropyLoss()
    for name, factory, cfg in NEIGHBOURS:
        torch.manual_seed(123)
        model = getattr(ref_models, factory)(**cfg)
        for mod in model.modules():                 # dropout draws depend on the dtype: switched off for this fixture
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
        # leave the vacuous default state (last-BN gamma = 0 silences whole branches): deterministic non-zero affine
        g = torch.Generator().manual_seed(99)
        with torch.no_grad():
            for n, p in model.named_parameters():
                if p.dim() == 1 and ('bn' in n or n.split('.')[-2].isdigit() or 'downsample' in n) and n.endswith('weight'):
                    p.copy_((0.5 + torch.rand(p.shape, generator=g)).to(torch.bfloat16).float())
        init = {k: v.clone() for k, v in model.state_dict().items()}
        model.double()                  # fp64: the comparison with the restatement is then free of rounding noise
        model.train()
        out = model(x.double())
        loss = crit(out, y)
        loss.backward()
        seen, names, norms = set(), [], []
        for n, p in model.named_parameters():          # named_parameters() lists a shared SE gate once
            if id(p) in seen or p.grad is None:
                continue
            seen.add(id(p)); names.append(n); norms.append(float(p.grad.norm()))
        stats = {k: float(v.double().sum()) for k, v in model.state_dict().items() if 'running_' in k}
        blob[name + '/logits'] = out.detach().numpy()
        blob[name + '/loss'] = np.float64(float(loss))
        blob[name + '/grad_names'] = np.array(names)
        blob[name + '/grad_norms'] = np.array(norms)
        blob[name + '/stat_names'] = np.array(list(stats.keys()))
        blob[name + '/stat_sums'] = np.array(list(stats.values()))
        # the perturbed affine parameters (everything else is re-created from the seed by the test)
        for k, v in init.items():
            if v.dim() == 1 and v.is_floating_point() and 'running' not in k and k.endswith('weight'):
                blob[name + '/affine/' + k] = bf16_bits(v)
        print(name, 'loss %.5f' % float(loss), '%d gradients' % len(names))
    np.savez_compressed(os.path.join(OUT, 'neighbours.npz'), **blob)
    print('neighbours fixture written')


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    ref_models, ref_trainer, ref_optim, ref_ce = import_reference()
    if len(sys.argv) > 1 and sys.argv[1] == 'neighbours':     # regenerate only this fixture
        neighbours_fixture(ref_models, ref_ce)
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'mobilenet_v2':   # regenerate only this fixture
        mobilenet_v2_fixture(ref_models, ref_trainer, ref_optim, ref_ce)
        return
    mobilenet_v2_fixture(ref_models, ref_trainer, ref_optim, ref_ce)

    # ---- 1. initialisation of the four model families under the CLI seed (main.py:114-115,137) ----
    init = {}
    for name, factory, cfg in [('resnet20_cifar10', ref_models.resnet, dict(dataset='cifar10', depth=20)),
                               ('resnet50_imagenet', ref_models.resnet, dict(dataset='imagenet', depth=50)),
                               ('resnext101_imagenet', ref_models.resnext, dict(dataset='imagenet', depth=101)),
                               ('mobilenet_v2', ref_models.mobilenet_v2, dict(dataset='imagenet')),
                               ('mobilenet_v1', ref_models.mobilenet, dict(dataset='imagenet'))]:
        torch.manual_seed(123)
        m = factory(**cfg)
        init[name] = {'stats': tensor_stats(m.state_dict()),
                      'n_params': sum(p.numel() for p in m.parameters())}
        if hasattr(m, 'regime'):
            init[name]['regime'] = [{k: (v if isinstance(v, (int, float, str)) else str(type(v).__name__))
                                     for k, v in ph.items()} for ph in m.regime]
    with open(os.path.join(OUT, 'init_stats.json'), 'w') as f:
        json.dump(init, f)
    if len(sys.argv) > 1 and sys.argv[1] == 'init':           # regenerate only the initialisation statistics
        return

    # ---- 2. resnet20: reference Trainer + OptimRegime, 5 warm-up steps then one recorded step ----
    torch.manual_seed(123)
    model = ref_models.resnet(dataset='cifar10', depth=20)
    x, y, rec = synth_record(8, (3, 32, 32), 10)
    crit = ref_ce.CrossEntropyLoss()
    opt = ref_optim.OptimRegime(model, model.regime)
    tr = ref_trainer.Trainer(model, crit, opt, device_ids=None, device='cpu', dtype=torch.float, print_freq=1000)
    model.train()
    losses = []
    for _ in range(5):
        _, loss, _ = tr._step(x, y, training=True)
        losses.append(float(loss))
    # the recorded step starts from this state with its parameters rounded to bf16, which the fixture then holds exactly
    # in half the bytes (the running statistics stay fp32), and from seeded momentum buffers
    mom_seed = 5
    mom_b = synthetic_momentum([(n, p.shape) for n, p in model.named_parameters()], mom_seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            p.copy_(p.to(torch.bfloat16).float())
            opt.optimizer.state[p]['momentum_buffer'].copy_(mom_b[n])
    state_b = deepcopy(model.state_dict())
    # recorded step: capture grads before the optimizer touches them
    opt.zero_grad(); opt.update(0, tr.training_steps)
    out = model(x); loss = crit(out, y); loss.backward()
    grads = {n: p.grad.clone() for n, p in model.named_parameters()}
    for p in model.parameters():
        p.grad.data.div_(1.0)
    opt.step()
    post = deepcopy(model.state_dict())
    blob = {**rec, 'logits': out.detach().numpy(), 'loss': np.float64(float(loss)), 'warm_losses': np.array(losses),
            'mom_seed': np.int64(mom_seed), 'mom_names': np.array([n for n, _ in model.named_parameters()])}
    for k, v in state_b.items():
        blob['state/' + k] = bf16_bits(v) if k in grads else v.numpy()
    # per parameter: the norm of its gradient, and the gradient and updated value at a fixed sample of elements
    rng = np.random.default_rng(0)
    for k, v in grads.items():
        idx = sample_index(v.numel(), rng)
        blob['idx/' + k] = idx
        blob['grad_norm/' + k] = np.float64(v.double().norm())
        blob['grad/' + k] = v.flatten().numpy()[idx]
        blob['post_norm/' + k] = np.float64(post[k].double().norm())
    for k, v in post.items():
        blob['post/' + k] = v.flatten().numpy()[blob['idx/' + k]] if k in grads else v.numpy()
    np.savez_compressed(os.path.join(OUT, 'resnet20_step.npz'), **blob)

    # ---- 3. reference Trainer.train loop over a tiny loader (loop-level golden) ----
    torch.manual_seed(123)
    model = ref_models.resnet(dataset='cifar10', depth=20)
    opt = ref_optim.OptimRegime(model, model.regime)
    tr = ref_trainer.Trainer(model, ref_ce.CrossEntropyLoss(), opt, device_ids=None, device='cpu',
                             dtype=torch.float, print_freq=1000)
    g = torch.Generator().manual_seed(7)
    batches = [(torch.randn(16, 3, 32, 32, generator=g), torch.randint(0, 10, (16,), generator=g)) for _ in range(4)]
    res = tr.train(batches)
    val = tr.validate(batches[:2])
    loop = {'train': {k: float(v) for k, v in res.items() if k in ('loss', 'prec1', 'prec5', 'error1', 'error5')},
            'val': {k: float(v) for k, v in val.items() if k in ('loss', 'prec1', 'prec5')},
            'training_steps': tr.training_steps, 'lr': opt.get_lr()[0]}
    post_stats = tensor_stats(model.state_dict())

    # ---- 4. resnet50 summary at a small size: 2 warm steps then a recorded step ----
    torch.manual_seed(123)
    model = ref_models.resnet(dataset='imagenet', depth=50)
    x50, y50, rec50 = synth_record(4, (3, 64, 64), 1000)
    opt = ref_optim.OptimRegime(model, model.regime)
    tr = ref_trainer.Trainer(model, ref_ce.CrossEntropyLoss(smooth_eps=0.1), opt, device_ids=None, device='cpu',
                             dtype=torch.float, print_freq=1000)
    model.train()
    l50 = []
    for _ in range(3):
        _, loss, _ = tr._step(x50, y50, training=True)
        l50.append(float(loss))
    opt.zero_grad()
    out = model(x50); loss = tr.criterion(out, y50); loss.backward()
    gn = {n: float(p.grad.norm()) for n, p in model.named_parameters()}
    np.savez(os.path.join(OUT, 'resnet50_summary.npz'), **rec50, logits=out.detach().numpy(),
             loss=np.float64(float(loss)), warm_losses=np.array(l50),
             grad_names=np.array(list(gn.keys())), grad_norms=np.array(list(gn.values())))

    # ---- 5. regimes: LR schedule, Mix&Match size table, sampled order ----
    reg = {}
    torch.manual_seed(123)
    m = ref_models.resnet(dataset='imagenet', depth=50, scale_lr=8, base_devices=8, base_device_batch=256)
    opt = ref_optim.OptimRegime(m, m.regime, log=False)
    sched = []
    for epoch, step in [(0, 0), (0, 1), (0, 300), (0, 1500), (2, 1251), (4, 3000), (5, 3200), (29, 18000),
                        (30, 18800), (60, 37600), (80, 50100), (89, 55000)]:
        opt.update(epoch, step)
        sched.append([epoch, step, opt.get_lr()[0]])
    reg['resnet50_scale8_lr'] = sched
    for mode in ('D+', 'B+'):
        torch.manual_seed(123)
        m = ref_models.resnet(dataset='imagenet', depth=50, regime='sampled', mix_size_regime=mode,
                              base_device_batch=256)
        reg['sampled_' + mode] = [[p, c] for p, c in m.sampled_data_regime]
        reg['sampled_regularizers'] = [r['name'] for r in m.regime[0]['regularizer']]
    torch.manual_seed(123)
    m = ref_models.resnet(dataset='cifar10', depth=20)
    opt = ref_optim.OptimRegime(m, m.regime, log=False)
    cif = []
    for epoch in (0, 80, 81, 121, 122, 164, 170):
        opt.update(epoch, epoch * 100)
        cif.append([epoch, opt.get_lr()[0]])
    reg['resnet20_lr'] = cif
    wd_names = [n for n, _ in opt.regularizer.regularization_list[0]._named_parameters]
    reg['resnet20_wd_params'] = wd_names
    with open(os.path.join(OUT, 'loop_and_regimes.json'), 'w') as f:
        json.dump({'loop': loop, 'loop_post_stats': post_stats, 'regimes': reg}, f)
    print('golden written to', OUT)


if __name__ == '__main__':
    main()
