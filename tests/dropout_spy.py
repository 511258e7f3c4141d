"""Test helper of the GPU dropout tests: see which dropout identity an op drew and which kernels it launched, and
rebuild the mask the kernels apply."""
import math

import torch


class Spy:
    """Records the dropout draws of ops._drop_args and the entry points called through lib.call."""

    def __init__(self, ops, monkeypatch):
        self.ops, self.mp, self.draws, self.calls = ops, monkeypatch, [], []
        orig_draw, orig_call = ops._drop_args, ops.lib.call

        def draw(*a):
            r = orig_draw(*a)
            self.draws.append(r)
            return r

        def call(name, *a):
            self.calls.append(name)
            return orig_call(name, *a)
        monkeypatch.setattr(ops, "_drop_args", draw)
        monkeypatch.setattr(ops.lib, "call", call)
        self.raw_call = orig_call

    def clear(self):
        self.draws.clear()
        self.calls.clear()


def rebuild_mask(spy, shape, p, seed_t, salt):
    """The kernels' dropout mask (0 or 1/(1-p)) of a tensor of ``shape`` for (p, seed, salt), as a CPU tensor."""
    ops = spy.ops
    ones = torch.ones(shape, device="cuda")
    m = torch.empty_like(ones)
    spy.raw_call("dv3_dropout", ops._p(ones), ops._p(m), ones.numel(), p, ops._p(seed_t), salt, ops._stream())
    m = m.cpu()
    kept = (m > 0).double().mean().item()
    n = m.numel()
    assert abs(kept - (1 - p)) <= 5 * math.sqrt(p * (1 - p) / n), (kept, p, n)      # dropout really on
    assert torch.all((m == 0) | (m == torch.tensor(1.0 / (1.0 - p), dtype=torch.float32)))
    return m
