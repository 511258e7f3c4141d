"""ops.convblock (Conv1dGLU / HighwayConv1d) with conv-input dropout on, in both arithmetic modes, against a float64
reference: output, dx and the weight-norm / bias gradients dv, dg, dbias.

The kernels regenerate the dropout mask of x from (seed, salt, flat (B,C,T) index) in several places: the forward
operand (tc: the split pass dv3_tc_split_input, whose planes the weight gradient reads as well; fp32: the convblock
loader and, separately, the dv3_conv1d_wgrad loader) and the data gradient's epilogue.  The test records the
(p, seed, salt) the call draws and rebuilds the mask with dv3_dropout on a (B,C,T) tensor of ones.  The reference
(modules.py:145-164, 200-226): xd = x * M, weight-normed conv of xd, GLU / highway gate, residual from the UNDROPPED x."""
import math

import pytest
import torch
import torch.nn.functional as F

import golden_util as G
from dropout_spy import Spy, rebuild_mask
from test_gpu_blocks import close, grad_close

pytestmark = pytest.mark.gpu
SEED = 0xD20F
# err(p > 0) <= 2 err(p = 0) + FLOOR (relative L2): an order of magnitude above the split-arithmetic error of a
# ConvBlock gradient and orders of magnitude below what a mask regenerated at a wrong index does.
DROP_RATIO, FLOOR = 2.0, 1e-4
GRADS = ("dx", "dv", "dg", "dbias")

# (math, B, C, T, k, dilation, causal, mode, residual)
SHAPES = [
    ("tc", 4, 256, 200, 3, 3, True, "glu", True),
    ("tc", 3, 128, 131, 5, 1, False, "hw", True),
    ("tc", 16, 512, 128, 3, 9, False, "glu", True),        # the benched encoder layer (deepvoice3_ljspeech, B = 16)
    ("fp32", 3, 64, 101, 3, 3, True, "glu", True),
    ("fp32", 2, 80, 77, 5, 1, False, "hw", True),
    ("fp32", 3, 80, 129, 3, 9, False, "glu", False),
]


def _inputs(B, C, T, k):
    gen = torch.Generator().manual_seed(B * 1000 + C + T + k)
    v = torch.randn(2 * C, C, k, generator=gen) * (4.0 / (k * C)) ** 0.5
    g = v.pow(2).sum((1, 2), keepdim=True).sqrt() * (1 + 0.2 * torch.randn(2 * C, 1, 1, generator=gen))
    bias = 0.1 * torch.randn(2 * C, generator=gen)
    x = torch.randn(B, C, T, generator=gen)
    return x, v, g, bias


def reference(x, v, g, bias, M, k, d, causal, mode, residual, R):
    """float64 forward + autograd -> {y, dx, dv, dg, dbias}."""
    x, v, g, bias = [t.double().requires_grad_(True) for t in (x, v, g, bias)]
    xd = x if M is None else x * M.double()
    w = g * v / v.pow(2).sum((1, 2), keepdim=True).sqrt()
    T = x.shape[2]
    pad = (k - 1) * d if causal else (k - 1) // 2 * d
    y = F.conv1d(xd, w, bias, padding=pad, dilation=d)[:, :, :T]
    a, b = y.split(y.shape[1] // 2, dim=1)
    s = torch.sigmoid(b)
    if mode == "glu":
        y = a * s
        if residual:
            y = (y + x) * math.sqrt(0.5)
    else:
        y = s * a + (1 - s) * x
    (y * R.double()).sum().backward()
    return {"y": y.detach(), "dx": x.grad, "dv": v.grad, "dg": g.grad, "dbias": bias.grad}


def _relerr(a, b):
    return float(torch.linalg.vector_norm(a.double() - b.double()) / torch.linalg.vector_norm(b.double()))


@pytest.fixture
def spy(monkeypatch):
    from deepvoice3_pytorch_b200 import ops
    return Spy(ops, monkeypatch)


def run(spy, math_mode, B, C, T, k, d, causal, mode, residual, p):
    ops = spy.ops
    spy.mp.setattr(ops, "conv_math", math_mode)
    x, v, g, bias = _inputs(B, C, T, k)
    xc, vc, gc, bc = [t.cuda().requires_grad_(True) for t in (x, v, g, bias)]
    R = G.loss_weights((B, C, T), 0)
    ops.rng.manual_seed(SEED, xc.device)
    ops.rng.start_forward()
    spy.clear()
    y = ops.convblock(xc, vc, gc, bc, None, k, d, causal, ops.MODE_GLU if mode == "glu" else ops.MODE_HIGHWAY,
                      residual, p_drop=p, training=True)
    (y * R.cuda()).sum().backward()
    torch.cuda.synchronize()
    if math_mode == "tc":
        assert {"dv3_tc_split_input", "dv3_tc_convblock_fwd", "dv3_tc_wgrad_mn"} <= set(spy.calls), spy.calls
    else:
        assert {"dv3_convblock_fwd", "dv3_conv1d_dgrad", "dv3_conv1d_wgrad"} <= set(spy.calls), spy.calls
        assert not any(c.startswith("dv3_tc_") for c in spy.calls), spy.calls
    assert len(spy.draws) == 1
    p_eff, seed_t, salt = spy.draws[0]
    M = rebuild_mask(spy, (B, C, T), p_eff, seed_t, salt) if p_eff > 0 else None
    ref = reference(x, v, g, bias, M, k, d, causal, mode, residual, R)
    got = {"y": y.detach().cpu(), "dx": xc.grad.cpu(), "dv": vc.grad.cpu(), "dg": gc.grad.cpu(), "dbias": bc.grad.cpu()}
    close(got["y"], ref["y"].numpy(), what="y p=%g" % p)
    for t in GRADS:
        grad_close(got[t], ref[t].numpy(), what="%s p=%g" % (t, p))
    return {t: _relerr(got[t], ref[t]) for t in got}


@pytest.mark.parametrize("math_mode,B,C,T,k,d,causal,mode,residual", SHAPES)
def test_convblock_dropout_vs_float64(math_mode, B, C, T, k, d, causal, mode, residual, spy):
    if math_mode == "tc":
        assert spy.ops.tc_supported(B, C, T, k), "shape must run on the tensor-core path"
    cfg = (math_mode, B, C, T, k, d, causal, mode, residual)
    err0 = run(spy, *cfg, 0.0)
    for p in (0.05, 0.5):
        err = run(spy, *cfg, p)
        for t, e in err.items():
            assert e <= DROP_RATIO * err0[t] + FLOOR, ("p=%g" % p, t, e, err0[t])
