"""Storage of large reference tensors in the golden files: a fixed, seeded sample of their elements.

A golden file keeps every element of small tensors.  A large tensor `key` is kept as the 1-D array of its elements at
sample_index(key, ...) (same dtype as the full tensor would have had), plus "shape:<key>" and "absmax:<key>" (the abs-max of
the WHOLE tensor, so that an error measured at the sampled positions is still normalised like max|t - ref| / max|ref|).
The positions are a function of the key alone, so the tests pick the same elements out of the tensor they compute."""
import zlib

import numpy as np
import torch


def sample_index(key, numel, n):
    """Sorted flat positions of the n elements of a `numel`-element tensor that are kept under `key`."""
    if n >= numel:
        return np.arange(numel)
    g = np.random.Generator(np.random.PCG64([31, zlib.crc32(key.encode())]))
    return np.sort(g.choice(numel, size=n, replace=False))


def keep_samples(out, sizes):
    """Replace each out[key] (a numpy array) named in sizes = {key: n} by its sample of n elements; record shape and abs-max."""
    for key, n in sizes.items():
        a = np.asarray(out[key])
        out["shape:" + key] = np.asarray(a.shape, np.int64)
        out["absmax:" + key] = np.asarray(np.abs(a.astype(np.float64)).max())
        out[key] = a.reshape(-1)[sample_index(key, a.size, n)]


def shape(gold, key):
    """Shape of the reference tensor `key`, sampled or not."""
    return tuple(int(s) for s in gold["shape:" + key]) if "shape:" + key in gold else tuple(gold[key].shape)


def absmax(gold, key):
    """Abs-max of the whole reference tensor `key`, sampled or not."""
    return float(gold["absmax:" + key]) if "absmax:" + key in gold else float(np.abs(gold[key].astype(np.float64)).max())


def at_sample(t, gold, key):
    """(t at the positions kept of `key`, the kept reference values) as flat float32 CPU tensors; t must have the stored shape.
    A tensor the file keeps whole is compared whole."""
    ref = np.asarray(gold[key])
    t = torch.as_tensor(t).detach().float().cpu()
    assert tuple(t.shape) == shape(gold, key), (key, tuple(t.shape), shape(gold, key))
    idx = torch.from_numpy(sample_index(key, t.numel(), ref.size))
    return t.reshape(-1)[idx], torch.from_numpy(ref.astype(np.float32)).reshape(-1)


def rel_max(t, gold, key):
    """max |t - ref| over the kept positions / max |ref| over the whole reference tensor."""
    a, r = at_sample(t, gold, key)
    return ((a - r).abs().max() / absmax(gold, key)).item()


def rel_l2(t, gold, key):
    """|t - ref| / |ref| (2-norms) over the kept positions."""
    a, r = at_sample(t, gold, key)
    return ((a - r).norm() / (r.norm() + 1e-30)).item()
