#!/usr/bin/env python
"""North-star benchmark: ResNet-50 training images/sec on synthetic 224x224 batches (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo's B200 kernel path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU trainer path (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's results to DIR/*.npy

One "step" = one full pass of the hot path over one batch: zero_grad -> forward -> CE loss -> backward ->
(all-reduce) -> fused SGD step, batch 256 per GPU, bf16 compute / fp32 masters.  Prints ONE JSON line
(rank 0).  ``value`` is the whole-job device-resident throughput, ``e2e`` the same metric through the
public API (Trainer) with pinned HOST batches: H2D of every batch and D2H of the loss inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

IMG = 224
CLASSES = 1000
# algorithmic work of one ResNet-50 training step per image (SURVEY.md section 8d): conv MACs fwd 4.0871 G;
# train = fprop + dgrad + wgrad, no dgrad for the stem  => 24.287 GFLOP/img
TRAIN_CONV_GFLOP_PER_IMG = 24.287


def parse():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=20)
    p.add_argument('--warmup', type=int, default=5)
    p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    p.add_argument('--batch', type=int, default=256, help='per-GPU batch')
    p.add_argument('--depth', type=int, default=50)
    p.add_argument('--model', default='resnet', choices=['resnet', 'resnext', 'mobilenet_v2'],
                   help='extra configurations (BASELINE configs[2..4]); the contract line is the default resnet-50')
    p.add_argument('--size', type=int, default=IMG, help='input resolution (Mix&Match sweep: 128..288)')
    p.add_argument('--no-e2e', action='store_true')
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--cpu-batch', type=int, default=32)
    p.add_argument('--dump-outputs', metavar='DIR', default=None,
                   help='after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32): '
                        'logits, loss, the updated parameters and the BatchNorm running statistics (a fixed sample of '
                        'an array larger than 16 MB)')
    args = p.parse_args()
    if args.steps < 1:
        p.error('--steps must be at least 1 (the number of timed steps)')
    return args


DUMP_MAX_ELEMS = 1 << 22   # per array: 16 MB of float32, so that the four arrays of a dump stay under 64 MB


def dump_outputs(path, arrays):
    """Write each tensor as path/<name>.npy in float32.  A tensor larger than DUMP_MAX_ELEMS is replaced by a fixed
    sample of its flattened elements (seed 0, ascending index order), identical from run to run for the same shape."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.flatten()[idx.to(t.device)]
        np.save(os.path.join(path, name + '.npy'), t.cpu().numpy())


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            d = json.load(f)
        return {'hbm_gbs': d['hbm_gbs'], 'tflops_burst': d['bf16_tflops'],
                'tflops': d.get('bf16_tflops_sustained', d['bf16_tflops']), 'source': 'measured'}
    except Exception:
        return {'hbm_gbs': 6650.0, 'tflops_burst': 1590.0, 'tflops': 1400.0, 'source': 'fallback'}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                f = [t.strip() for t in out.stdout.strip().split(',')]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unsampled']}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith('active') for s in self.samples)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.samples[0][1]), 'reasons': reasons,
                'power_w_max': max(float(s[2]) for s in self.samples), 'samples': len(self.samples)}


def default_cfg_for_traffic(args):
    return args.model == 'resnet' and args.depth == 50 and args.size == IMG and args.batch == 256


def usable_cores():
    """host threads this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def cpu_reference(batch, steps, warmup, depth):
    """The reference's CPU trainer path (oracle port of models/resnet.py + Trainer._step + OptimRegime.step),
    fp32, all host threads, on a bounded sample of the workload (batch ``batch`` instead of 256)."""
    from oracle import ref_model
    from convnet.pytorch_b200 import models
    torch.set_num_threads(int(os.environ.get('B200_CPU_THREADS', usable_cores())))
    torch.manual_seed(123)
    sd = {k: v.clone() for k, v in models.resnet(dataset='imagenet', depth=depth).state_dict().items()}
    g = torch.Generator().manual_seed(0)
    x = torch.randn(batch, 3, IMG, IMG, generator=g)
    y = torch.randint(0, CLASSES, (batch,), generator=g)
    mom = {}
    t0 = None
    for i in range(warmup + steps):
        if i == warmup:
            t0 = time.perf_counter()
        _, loss, grads, bufs = ref_model.loss_and_grads(sd, x, y)
        sd, mom = ref_model.sgd_step(sd, grads, mom, lr=0.1)
        sd.update(bufs)
    dt = time.perf_counter() - t0
    return {'value': batch * steps / dt, 'unit': 'images/sec', 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': 'ResNet-%d fp32 CPU, batch %d (of 256) x %d steps after %d warm-up, %.2f s/step'
                      % (depth, batch, steps, warmup, dt / steps), 'ms_per_step': 1e3 * dt / steps}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warm = 1
    cb = cpu_reference(args.cpu_batch, steps, warm, args.depth)
    line = {'impl': 'reference', 'metric': 'ResNet-50 images/sec (training step, synthetic 224x224)',
            'value': cb['value'], 'unit': 'images/sec', 'n_gpus': args.gpus, 'steps': steps, 'warmup': warm,
            'ms_per_step': cb['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'ResNet-%d, synthetic ImageNet 224x224, SGD+momentum+WD, reference CPU trainer '
                                   'path on host cores; bounded sample: batch %d' % (args.depth, args.cpu_batch),
                       'global_batch': args.cpu_batch, 'parallelism': 'cpu'},
            'cpu_baseline': {k: cb[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
            'e2e': {'value': cb['value'], 'unit': 'images/sec', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the B200 path has no CPU fallback '
                         '(use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    distributed = world > 1
    if distributed:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    from convnet.pytorch_b200 import models, lib, ops
    from convnet.pytorch_b200.engine import convert_b200
    from convnet.pytorch_b200.trainer import Trainer
    from convnet.pytorch_b200.utils.optim import OptimRegime
    from convnet.pytorch_b200.utils.cross_entropy import CrossEntropyLoss

    B = args.batch
    torch.manual_seed(123)
    if args.model == 'mobilenet_v2':
        model = models.mobilenet_v2(dataset='imagenet')
    else:
        model = getattr(models, args.model)(dataset='imagenet', depth=args.depth)
    convert_b200(model, dev)
    criterion = CrossEntropyLoss().to(dev)
    optimizer = OptimRegime(model, model.regime)
    trainer = Trainer(model, criterion, optimizer, device_ids=[local], device=str(dev), dtype=torch.float,
                      distributed=distributed, local_rank=local, print_freq=10 ** 9)
    g = torch.Generator().manual_seed(rank)            # per-rank data (DistributedSampler analogue)
    x_host = torch.randn(B, 3, args.size, args.size, generator=g).pin_memory()
    y_host = torch.randint(0, CLASSES, (B,), generator=g).pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)
    model.train()

    def sync_all():
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
            torch.cuda.synchronize()

    def device_step():
        # same sequence as Trainer._step (trainer.py:106-177) with the batch already resident in HBM
        optimizer.zero_grad()
        optimizer.update(0, trainer.training_steps)
        replayed = trainer.graphed_forward_backward(x_dev, y_dev)   # CUDA-graph replay once the shape is warm
        if replayed is None:
            out = model(x_dev)
            loss = criterion(out, y_dev)
            loss.backward()
        else:
            out, loss = replayed[0], replayed[1]
        trainer._allreduce_gradients()
        optimizer.set_grad_unscale(1.0, world)
        optimizer.step()
        trainer.training_steps += 1
        return out, loss

    for _ in range(max(args.warmup, 4)):   # steps 1-2 eager, 3 captures the CUDA graph, 4+ replay it
        device_step()
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = lib.launch_count() + trainer.graph_replayed_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_enq = time.perf_counter()
    for _ in range(args.steps):
        out, loss = device_step()
    e1.record()
    enqueue_ms = (time.perf_counter() - t_enq) * 1e3 / args.steps     # host time to launch one step (no syncs)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = lib.launch_count() + trainer.graph_replayed_launches - launches0
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    clocks = sampler.stop() if sampler else None
    final_loss = float(loss.detach())
    if args.dump_outputs and rank == 0:
        # before the e2e windows below train the model further
        dump_outputs(args.dump_outputs, {
            'logits': out, 'loss': loss.reshape(1),
            'params': torch.cat([p.detach().flatten() for p in model.parameters()]),
            'bn_running_stats': torch.cat([b.detach().float().flatten() for n, b in model.named_buffers()
                                           if 'running' in n])})
    sync_all()

    # ---- end to end through the public API: pinned host batches, H2D + loss D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        loader = [(x_host, y_host)] * 2
        trainer.forward(loader, training=True)           # warm the path
        sync_all()
        n_e2e = max(10, args.steps)
        # raw pinned-host -> device bandwidth of this box (explains e2e when PCIe, not the GPU, is the bound)
        h2d_ms = float('inf')
        x_probe = torch.empty_like(x_dev)
        for _ in range(3):            # best of 3 into a preallocated buffer (the first copy pays one-off set-up)
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            x_probe.copy_(x_host, non_blocking=True)
            h1.record()
            torch.cuda.synchronize()
            h2d_ms = min(h2d_ms, h0.elapsed_time(h1))
        del x_probe
        loader = [(x_host, y_host)] * n_e2e
        windows = []
        for _ in range(3):    # three windows of n_e2e steps; the first one still pays one-off allocator / replay warm-up
            t0 = time.perf_counter()
            res = trainer.forward(loader, training=True)
            torch.cuda.synchronize()
            windows.append(time.perf_counter() - t0)
        dt = torch.tensor([min(windows)], device=dev, dtype=torch.float64)
        if distributed:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        # (f2) device input pipeline: uint8 NHWC host batches (what an image decoder yields), normalised by the stem's
        # relayout kernel -- 4x fewer PCIe bytes than the fp32 NCHW batch of the reference's loader contract
        u8 = None
        try:
            xu8 = torch.randint(0, 256, (B, args.size, args.size, 3), dtype=torch.uint8).pin_memory()
            loader8 = [(xu8, y_host)] * n_e2e
            trainer.forward(loader8[:4], training=True)
            sync_all()
            t0 = time.perf_counter()
            trainer.forward(loader8, training=True)
            torch.cuda.synchronize()
            d8 = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if distributed:
                dist.all_reduce(d8, op=dist.ReduceOp.MAX)
            u8 = {'value': world * B * n_e2e / float(d8), 'unit': 'images/sec',
                  'h2d_bytes_per_step': xu8.numel() + y_host.numel() * 8, 'd2h_bytes_per_step': 12,
                  'input': 'uint8 NHWC + on-device normalisation (b200_input_prep_u8)'}
        except Exception as exc:  # noqa: BLE001
            u8 = {'error': str(exc)[:200]}
        sync_all()
        e2e = {'value': world * B * n_e2e / float(dt), 'unit': 'images/sec', 'uint8_input': u8,
               'h2d_bytes_per_step': x_host.numel() * 4 + y_host.numel() * 8,
               'd2h_bytes_per_step': 4 + 2 * 4, 'steps': n_e2e,
               'windows_ms_per_step': [round(1e3 * w / n_e2e, 3) for w in windows], 'window_policy': 'min of 3',
               'h2d_gbs_measured': x_host.numel() * 4 / h2d_ms / 1e6,
               'host_enqueue_ms_per_step': enqueue_ms, 'host_cores': usable_cores(),
               'api': 'Trainer.forward(loader, training=True): H2D of the fp32 NCHW batch (side stream, one step ahead) + '
                      'asynchronous read-back of {loss, prec1, prec5} every step'}
        sync_all()

    # ---- per-kernel-class device time of one extra step (CUDA events around every library call) ----
    roof = None
    trainer.use_graphs = False   # eager launches so that every library call can be bracketed by CUDA events
    model._b200._wg_stream = None   # ... and on ONE stream (the wgrad side stream would overlap the classes)
    ops.start_timing()      # every rank runs the step (it contains the gradient all-reduce); rank 0 reports
    device_step()
    torch.cuda.synchronize()
    classes = ops.stop_timing()
    sync_all()
    if rank == 0:
        pk = peaks()
        total_ms = sum(c['ms'] for c in classes.values())
        conv_names = [n for n in classes if n.startswith('conv_')]
        conv_ms = sum(classes[n]['ms'] for n in conv_names)
        conv_flops = sum(classes[n]['flops'] for n in conv_names)
        hbm_names = [n for n in classes if not n.startswith('conv_') and n != 'allreduce_nccl']
        hbm_ms = sum(classes[n]['ms'] for n in hbm_names)
        hbm_bytes = sum(classes[n]['bytes'] for n in hbm_names)
        # the gradient all-reduce is not one of this library's kernels and its first eager call is not steady state:
        # it is reported under 'classes' but never picked as the dominant kernel
        dom = max((n for n in classes if n != 'allreduce_nccl'), key=lambda n: classes[n]['ms'])
        d = classes[dom]
        if dom.startswith('conv_'):
            ach = d['flops'] / (d['ms'] * 1e-3) / 1e12 / max(d['calls'], 1) * d['calls']
            roof = {'kernel': dom, 'bound': 'tensor', 'achieved': ach, 'peak': pk['tflops'], 'unit': 'TFLOP/s',
                    'frac': ach / pk['tflops'], 'traffic': None}
        else:
            ach = d['bytes'] / (d['ms'] * 1e-3) / 1e9
            roof = {'kernel': dom, 'bound': 'hbm', 'achieved': ach, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                    'frac': ach / pk['hbm_gbs'], 'traffic': None}
        # traffic: DRAM bytes (ncu dram__bytes_read.sum + dram__bytes_write.sum) per launch of the dominant class, from
        # the committed launch list of this same command (profiles/r02_traffic.json; tools/profile_round2.sh)
        try:
            with open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')) as f:
                tj = json.load(f)['classes']
            key = dom if dom in tj else ('conv_fprop+dgrad' if dom in ('conv_fprop', 'conv_dgrad') else None)
            if key and default_cfg_for_traffic(args):
                roof['traffic'] = (tj[key]['dram_read_bytes'] + tj[key]['dram_write_bytes']) / max(tj[key]['launches'], 1)
                roof['traffic_unit'] = 'bytes per launch (class average; ncu, profiles/r02_traffic.json)'
                roof['algorithmic_bytes_per_launch'] = d['bytes'] / max(d['calls'], 1) if d.get('bytes') else None
        except Exception:
            pass
        roof['peak_source'] = pk['source'] + (' sustained' if dom.startswith('conv_') else '')
        roof['launches_of_kernel_per_step'] = d['calls']
        roof['avg_launch_ms'] = d['ms'] / max(d['calls'], 1)
        roof['step_share'] = d['ms'] / total_ms if total_ms else None
        roof['conv_all'] = {'tflops': conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms else None,
                            'frac_of_tensor_peak': conv_flops / (conv_ms * 1e-3) / 1e12 / pk['tflops'] if conv_ms else None,
                            'ms': conv_ms}
        roof['hbm_all'] = {'gbs': hbm_bytes / (hbm_ms * 1e-3) / 1e9 if hbm_ms else None,
                           'frac_of_hbm_peak': hbm_bytes / (hbm_ms * 1e-3) / 1e9 / pk['hbm_gbs'] if hbm_ms else None,
                           'ms': hbm_ms}
        roof['classes'] = {n: {'ms': round(c['ms'], 3), 'calls': c['calls']} for n, c in sorted(classes.items())}

    cpu_base = None
    default_cfg = args.model == 'resnet' and args.depth == 50 and args.size == IMG
    if rank == 0 and world == 1 and not args.no_cpu_baseline and default_cfg:
        cb = cpu_reference(args.cpu_batch, 3, 1, args.depth)
        cpu_base = {k: cb[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}

    if rank == 0:
        ips = world * B * args.steps / (ms * 1e-3)
        name = {'resnet': 'ResNet-%d', 'resnext': 'ResNeXt-%d 32x4d', 'mobilenet_v2': 'MobileNet-v2'}[args.model]
        name = name % args.depth if '%d' in name else name
        line = {'metric': '%s images/sec (training step, synthetic %dx%d)' % (name, args.size, args.size), 'value': ips,
                'unit': 'images/sec', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 4),
                'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16', 'data': 'synthetic',
                'config': {'workload': '%s bf16 (fp32 master weights), synthetic ImageNet %dx%d, batch %d/GPU, '
                                       'SGD momentum 0.9 + WeightDecay 1e-4%s'
                                       % (name, args.size, args.size, B,
                                          ' (BASELINE.json configs[1])' if default_cfg else ''),
                           'global_batch': world * B, 'parallelism': 'dp%d' % world,
                           'l2_policy': 'per-step working set (activations ~10 GB) >> 126 MB L2; no explicit flush'},
                'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches, 'roofline': roof, 'cpu_baseline': cpu_base,
                'final_loss': final_loss,
                'conv_tensor_pipe_frac': (world * B * args.steps * TRAIN_CONV_GFLOP_PER_IMG / (ms * 1e-3) / 1e3
                                          / (world * peaks()['tflops'])) if default_cfg else None}
        print(json.dumps(line), flush=True)
    if distributed:
        shutdown(trainer)


def shutdown(trainer):
    """Leave a multi-rank run promptly: captured graphs released first (they hold NCCL work), then barrier + destroy, with
    a watchdog that hard-exits if the teardown blocks (the JSON line is already printed and flushed)."""
    def _bail():
        sys.stdout.flush()
        os._exit(0)
    timer = threading.Timer(20.0, _bail)
    timer.daemon = True
    timer.start()
    trainer.release_graphs()
    dist.barrier()
    dist.destroy_process_group()
    # the result line is out and every rank passed the barrier: skip interpreter finalisation (communicator / context
    # destructors have been seen to block after graphs with captured collectives) -- the timer stays armed until here
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
