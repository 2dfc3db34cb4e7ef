"""CPU-side checks: the C-ABI library loads and exports every symbol of include/b200conv.h, the binding
covers the header, the product path fails loudly without CUDA (no CPU fallback), regime / data-regime host
logic, and the N>1 gradient reduction logic under gloo (world_size 2)."""
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, 'include', 'b200conv.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(b200_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    from convnet.pytorch_b200 import lib
    assert lib.available(), 'libb200conv.so missing: run __graft_entry__.build()'
    handle = lib.load()
    names = _header_functions()
    assert len(names) >= 25
    for n in names:
        assert hasattr(handle, n), 'symbol %s declared in include/b200conv.h is not exported' % n
    assert sorted(lib.SIGNATURES) == names, 'ctypes binding and header disagree'
    assert handle.b200_version() >= 100
    assert handle.b200_launch_count() == 0 or handle.b200_launch_count() > 0


def test_product_path_fails_loudly_without_cuda():
    from convnet.pytorch_b200 import models, ops
    from convnet.pytorch_b200.engine import convert_b200
    from convnet.pytorch_b200.lib import B200Error
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    m = models.resnet(dataset='cifar10', depth=20)
    with pytest.raises(B200Error):
        convert_b200(m)
    with pytest.raises(B200Error):
        ops.bn_apply(torch.zeros(8, 8, dtype=torch.bfloat16), torch.ones(8), torch.zeros(8))
    with pytest.raises(B200Error):
        models.resnet(dataset='cifar10', depth=20, b200=True)


def test_no_product_module_imports_the_oracle():
    pkg = os.path.join(ROOT, 'convnet')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, flags=re.M), os.path.join(dirpath, f)


def test_regime_grammar():
    from convnet.pytorch_b200.utils.regime import Regime
    hits = []
    r = Regime([{'epoch': 0, 'lr': 1.0, 'k': 'a'}, {'epoch': 2, 'lr': 0.5, 'execute_once': lambda: hits.append(1)},
                {'step': 100, 'step_lambda': "lambda t: {'lr': 0.1 * t}"}], {})
    assert r.update(0, 0) and r.setting['lr'] == 1.0
    assert not r.update(1, 10)
    assert r.update(2, 20) and r.setting['lr'] == 0.5 and r.setting['k'] == 'a' and hits == [1]
    r.update(2, 21)
    assert hits == [1]
    assert r.update(2, 100) and abs(r.setting['lr'] - 10.0) < 1e-12
    assert r.update(2, 101) and abs(r.setting['lr'] - 10.1) < 1e-12


def test_data_regime_synthetic_and_sampled():
    from convnet.pytorch_b200.data import DataRegime, SampledDataRegime
    d = DataRegime([{'epoch': 0, 'input_size': 32, 'batch_size': 8}, {'epoch': 1, 'batch_size': 4}],
                   defaults={'name': 'synthetic_cifar10', 'split': 'train', 'synthetic_length': 64, 'shuffle': False,
                             'drop_last': True})
    x, y = next(iter(d.get_loader()))
    assert x.shape == (8, 3, 32, 32) and y.dtype == torch.int64 and len(d) == 64
    d.set_epoch(1)
    assert next(iter(d.get_loader()))[0].shape[0] == 4
    regs = [DataRegime(None, defaults={'name': 'synthetic_imagenet', 'split': 'train', 'synthetic_length': 48,
                                       'input_size': s, 'batch_size': b, 'duplicates': dup, 'drop_last': True})
            for s, b, dup in ((32, 4, 2), (64, 2, 1))]
    sam = SampledDataRegime(regs, [0.5, 0.5])
    sam.set_epoch(0)
    shapes = [tuple(x.shape) for x, _ in sam.get_loader()]
    assert (4, 2, 3, 32, 32) in shapes and (2, 3, 64, 64) in shapes
    assert shapes == [tuple(x.shape) for x, _ in sam.get_loader()]  # epoch-seeded order: identical on every rank


def test_trainer_duplicates_and_chunks_cpu():
    from convnet.pytorch_b200 import models
    from convnet.pytorch_b200.trainer import Trainer, _flatten_duplicates
    from convnet.pytorch_b200.utils.optim import OptimRegime
    from convnet.pytorch_b200.utils.cross_entropy import CrossEntropyLoss
    x = torch.arange(2 * 3 * 1 * 2 * 2, dtype=torch.float).view(2, 3, 1, 2, 2)
    fx, fy = _flatten_duplicates(x, torch.tensor([5, 7]))
    assert fx.shape == (6, 1, 2, 2) and fy.tolist() == [5, 5, 5, 7, 7, 7]
    torch.manual_seed(0)
    model = models.resnet(dataset='cifar10', depth=8)
    tr = Trainer(model, CrossEntropyLoss(), OptimRegime(model, model.regime), device_ids=None, device='cpu',
                 print_freq=1000, grad_clip=1.0)
    batches = [(torch.randn(4, 2, 3, 32, 32), torch.randint(0, 10, (4,))) for _ in range(2)]
    res = tr.train(batches, chunk_batch=2)
    assert tr.training_steps == 2 and 'grad' in res and res['loss'] > 0


def _gloo_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from convnet.pytorch_b200 import models
    from convnet.pytorch_b200.trainer import Trainer
    from convnet.pytorch_b200.utils.optim import OptimRegime
    from convnet.pytorch_b200.utils.cross_entropy import CrossEntropyLoss
    torch.manual_seed(123 + rank)          # different init per rank: the ctor broadcast must fix it
    model = models.resnet(dataset='cifar10', depth=8)
    tr = Trainer(model, CrossEntropyLoss(), OptimRegime(model, model.regime), device_ids=None, device='cpu',
                 distributed=True, local_rank=rank, print_freq=1000)
    g = torch.Generator().manual_seed(rank)
    batches = [(torch.randn(8, 3, 32, 32, generator=g), torch.randint(0, 10, (8,), generator=g)) for _ in range(2)]
    tr.train(batches)
    flat = torch.cat([p.detach().flatten() for p in model.parameters()])
    gathered = [torch.zeros_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    same = all(torch.equal(gathered[0], t) for t in gathered)

    # arena-style reduction used by the B200 path: sum all-reduce + 1/world folded into the optimizer scale
    class _Arena:
        g32 = torch.full((10,), float(rank + 1))
    class _RT:
        arena = _Arena()
        grad_bucket_hook = None
    tr.b200, tr.world_size = _RT(), world
    tr._allreduce_gradients()
    # bucketed form (what the backward pass drives on the B200 path): ranges reduced as they become final, in
    # reverse arena order, must add up to the same flat sum; afterwards _allreduce_gradients has nothing left to do
    class _Arena2:
        g32 = torch.arange(12, dtype=torch.float32) * (rank + 1)
    hook = Trainer._GradBuckets(_Arena2, 'cpu')
    for lo, hi in ((8, 12), (3, 8), (0, 3)):
        hook.bucket(lo, hi, None)
    hook.finish()
    _RT.grad_bucket_hook = hook
    tr._allreduce_gradients()
    ok_buckets = bool(torch.equal(_Arena2.g32, torch.arange(12, dtype=torch.float32) * sum(range(1, world + 1)))) \
        and hook.launched == 3 and bool(torch.all(_Arena.g32 == sum(range(1, world + 1))))
    opt = OptimRegime(models.resnet(dataset='cifar10', depth=8), [{'epoch': 0, 'optimizer': 'SGD', 'lr': 0.1}])
    opt.set_grad_unscale(4.0, world)
    ok_sum = bool(torch.all(_Arena.g32 == sum(range(1, world + 1)))) and abs(opt._inv_scale - 1.0 / (4.0 * world)) < 1e-12
    if rank == 0:
        ret['same'], ret['sum'] = same, ok_sum and ok_buckets
    dist.destroy_process_group()


def test_data_parallel_world2_gloo():
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29500 + os.getpid() % 2000
    mp.spawn(_gloo_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret['same'], 'parameters diverged across ranks'
    assert ret['sum'], 'flat-arena all-reduce / folded 1/world factor wrong'


def test_cli_cpu_plumbing_run(tmp_path):
    """BASELINE config C1 through the reference-compatible CLI (main.py:28-360 of the reference): resnet depth 20 on
    synthetic CIFAR-10, CPU, stock torch layers: train -> validate -> checkpoint -> results.csv."""
    from convnet.pytorch_b200 import main as cli
    cli.main(['--model', 'resnet', '--model-config', "{'depth': 20}", '--dataset', 'synthetic_cifar10',
              '--device', 'cpu', '-b', '16', '--epochs', '1', '--max-steps', '3', '--workers', '0',
              '--results-dir', str(tmp_path), '--save', 'cli_cpu'])
    out = tmp_path / 'cli_cpu'
    for name in ('checkpoint.pth.tar', 'model_best.pth.tar', 'results.csv', 'config.json', 'log.txt'):
        assert (out / name).exists(), name
    import csv
    rows = list(csv.DictReader(open(out / 'results.csv')))
    assert len(rows) == 1 and float(rows[0]['training loss']) > 0 and 0 <= float(rows[0]['validation prec1']) <= 100
    ck = torch.load(out / 'checkpoint.pth.tar', map_location='cpu', weights_only=False)
    assert ck['epoch'] == 1 and 'state_dict' in ck and any(k.endswith('conv1.weight') for k in ck['state_dict'])


def test_evaluate_cli_cpu(tmp_path):
    """evaluate.py of the reference (evaluate.py:101-193): checkpoint -> [--absorb-bn] [--calibrate-bn] [--avg-out]
    -> validate.  CPU / torch-module form; absorbing BatchNorm must not change the metrics."""
    from convnet.pytorch_b200 import main as cli
    from convnet.pytorch_b200 import evaluate as ev
    cli.main(['--model', 'resnet', '--model-config', "{'depth': 8}", '--dataset', 'synthetic_cifar10',
              '--device', 'cpu', '-b', '16', '--epochs', '1', '--max-steps', '2', '--workers', '0',
              '--results-dir', str(tmp_path), '--save', 'run'])
    ck = str(tmp_path / 'run' / 'checkpoint.pth.tar')
    os.environ['B200_SYNTHETIC_LENGTH'] = '64'
    try:
        base = ev.main([ck, '--dataset', 'synthetic_cifar10', '--device', 'cpu', '-b', '16', '--workers', '0'])
        absorbed = ev.main([ck, '--dataset', 'synthetic_cifar10', '--device', 'cpu', '-b', '16', '--workers', '0',
                            '--absorb-bn'])
        both = ev.main([ck, '--dataset', 'synthetic_cifar10', '--device', 'cpu', '-b', '16', '--workers', '0',
                        '--absorb-bn', '--calibrate-bn', '--calibrate-steps', '2', '--avg-out', '--duplicates', '2'])
    finally:
        del os.environ['B200_SYNTHETIC_LENGTH']
    assert abs(base['loss'] - absorbed['loss']) < 1e-4 * max(1.0, base['loss']) and base['prec1'] == absorbed['prec1']
    assert both['loss'] > 0 and 0 <= both['prec1'] <= 100


def test_committed_profile_feeds_bench_traffic(tmp_path):
    """bench.py reports roofline.traffic from profiles/r02_traffic.json (DRAM bytes per launch of the dominant kernel
    class, produced by tools/summarize_launches.py from the committed ncu launch list profiles/r02_launches.csv): the
    file must carry the class bench.py looks up, and the summariser must reproduce it from that launch list, stored
    gzip-compressed as tests/golden/r02_launches.csv.gz."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, 'profiles', 'r02_traffic.json')) as f:
        tj = json.load(f)['classes']
    for key in ('conv_fprop+dgrad', 'conv_wgrad', 'bn_apply', 'bn_bwd_dx', 'bn_bwd_reduce'):
        assert tj[key]['launches'] > 0 and tj[key]['dram_read_bytes'] > 0, key
    out_md, out_js = str(tmp_path / 'r02_launches_check.md'), str(tmp_path / 'r02_traffic_check.json')
    r = subprocess.run([sys.executable, os.path.join(root, 'tools', 'summarize_launches.py'),
                        os.path.join(root, 'tests', 'golden', 'r02_launches.csv.gz'), out_md, 'check', out_js],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-500:]
    with open(out_js) as f:
        again = json.load(f)['classes']
    assert again['conv_fprop+dgrad']['launches'] == tj['conv_fprop+dgrad']['launches']
    assert abs(again['conv_fprop+dgrad']['dram_read_bytes'] - tj['conv_fprop+dgrad']['dram_read_bytes']) < 1.0
    with open(out_md) as f:
        assert 'b200::conv_igemm_kernel' in f.read()

