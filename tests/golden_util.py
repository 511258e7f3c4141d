"""Reader and writer of the golden vectors under tests/golden/ (make_golden.py, make_train_golden.py,
make_dropin_golden.py)."""
import glob
import os
from collections import defaultdict

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SHARD_BYTES = 900000         # raw bytes per file, per-array zip / .npy headers included: every file stays under 1 MB
_cache = {}


def _shards(fname):
    stem = os.path.join(GOLDEN, fname[:-len(".npz")])
    return sorted(glob.glob(stem + ".*.npz"), key=lambda p: int(p.rsplit(".", 2)[1]))


def save(fname, arrays):
    """{"case|group|name": array} -> tests/golden/<stem>.<i>.npz, compressed; arrays go into the shards in order and a
    shard is closed before its raw size passes SHARD_BYTES."""
    for old in _shards(fname):
        os.remove(old)
    stem = os.path.join(GOLDEN, fname[:-len(".npz")])
    shards, size = [{}], 0
    for key, value in arrays.items():
        value = np.asarray(value)
        n = value.nbytes + 512
        if shards[-1] and size + n > SHARD_BYTES:
            shards.append({})
            size = 0
        shards[-1][key] = value
        size += n
    for i, shard in enumerate(shards):
        np.savez_compressed("%s.%d.npz" % (stem, i), **shard)
    total = sum(os.path.getsize(p) for p in _shards(fname))
    print("wrote %s: %d arrays in %d files, %.1f KB" % (fname, len(arrays), len(shards), total / 1024))


def load(fname):
    """-> {case: {group: {name: np.ndarray}}} of all shards of ``fname``"""
    if fname not in _cache:
        paths = _shards(fname)
        assert paths, "no golden shards for %s under %s" % (fname, GOLDEN)
        out = defaultdict(lambda: defaultdict(dict))
        for path in paths:
            z = np.load(path, allow_pickle=False)
            for key in z.files:
                case, group, name = key.split("|")
                out[case][group][name] = z[key]
        _cache[fname] = out
    return _cache[fname]


def tensors(d, device="cpu", dtype=None):
    out = {}
    for k, v in d.items():
        t = torch.from_numpy(np.ascontiguousarray(v))
        if dtype is not None and t.is_floating_point():
            t = t.to(dtype)
        out[k] = t.to(device)
    return out


def loss_weights(shape, i, device="cpu", dtype=torch.float32):
    """Same projection tensor as make_golden.loss_weights."""
    n = int(np.prod(shape))
    return torch.cos(torch.arange(n, dtype=torch.float64) * 0.37 + i).to(torch.float32) \
        .reshape(shape).to(device=device, dtype=dtype)


def meta_scalar(case, name):
    return case["meta"][name].item()


def kwargs_of(case):
    kw = {}
    for k, v in case["kw"].items():
        if v.dtype.kind in "US":
            kw[k] = str(v)
        elif v.dtype.kind == "b":
            kw[k] = bool(v)
        elif v.dtype.kind in "iu":
            kw[k] = int(v)
        else:
            kw[k] = float(v)
    return kw
