"""Encodings of the committed golden fixtures (tests/golden/*), shared by their generator (oracle/make_golden.py) and
the tests that read them.

Input batches are not stored: a fixture records the arguments of ``synth`` and a ``probe`` of the values, and the test
re-draws the batch and checks the probe.  Values that are bf16-exact are stored as their bf16 bits (uint16), in half
the bytes of fp32.  The recorded ResNet-20 step starts from momentum buffers drawn by ``synthetic_momentum`` from a seed
in an order the fixture stores by name.
"""
import numpy as np
import torch


def synth(batch, shape, classes, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, *shape, generator=g), torch.randint(0, classes, (batch,), generator=g)


def probe(x):
    """every 1021st element of the flattened batch: enough to tell whether a re-drawn batch is the stored one."""
    return x.flatten()[::1021].numpy()


def synth_record(batch, shape, classes, seed=0):
    """``synth`` plus what a fixture stores instead of the batch itself: the arguments and a probe of the values."""
    x, y = synth(batch, shape, classes, seed)
    return x, y, dict(x_shape=np.array([batch, *shape]), x_seed=np.int64(seed), n_classes=np.int64(classes),
                      x_probe=probe(x), y=y.numpy())


def redraw(z):
    """the input batch of a loaded fixture ``z``, re-drawn from its seed; raises if it is not the batch recorded."""
    shape = [int(n) for n in z['x_shape']]
    x, y = synth(shape[0], shape[1:], int(z['n_classes']), int(z['x_seed']))
    if not (np.array_equal(probe(x), z['x_probe']) and np.array_equal(y.numpy(), z['y'])):
        raise ValueError('the re-drawn input batch is not the one the fixture recorded')
    return x, y


def bf16_bits(t):
    """a tensor whose values are bf16-exact -> its bf16 bits (uint16)."""
    b = t.to(torch.bfloat16)
    assert torch.equal(b.float(), t.float())
    return b.view(torch.int16).numpy().view(np.uint16)


def decode(a):
    """fixture array -> fp32/int tensor; uint16 arrays are bf16 bits written by ``bf16_bits``."""
    return torch.from_numpy(a.view(np.int16)).view(torch.bfloat16).float() if a.dtype == np.uint16 else torch.from_numpy(a)


def synthetic_momentum(named_shapes, seed):
    """bf16-exact momentum buffers drawn from a seed, one per (name, shape) in the order given: the recorded ResNet-20
    step starts from these, so that the fixture need not hold a second copy of the network's size."""
    g = torch.Generator().manual_seed(seed)
    return {k: (1e-2 * torch.randn(s, generator=g)).to(torch.bfloat16).float() for k, s in named_shapes}
