"""ops.attention_core against a float64 reference (attention_cases.reference), forward and backward, with attention
dropout on, on both kernel paths: the fused tcgen05 kernels (csrc/tc_attn.cu) and the exact-fp32 SIMT kernels
(dv3_bgemm + dv3_softmax_*, fp32 mode and Ts > 128).

Every dropout site in csrc/ keeps element i of its tensor iff f(seed, salt, i): the test records the (p, seed, salt)
the call draws and rebuilds the mask M with dv3_dropout on a (B,Td,Ts) tensor of ones, so the reference applies the
mask the kernels must have regenerated in all three places (forward epilogue, softmax-backward epilogue, Pd staging
of the key/value-gradient kernel).  Error bounds: attention_cases.BOUNDS, calibrated by test_attention_tolerance.py."""
import math

import pytest
import torch

import attention_cases as A
from dropout_spy import Spy, rebuild_mask

pytestmark = pytest.mark.gpu
SEED = 0x5EED1234


@pytest.fixture
def spy(monkeypatch):
    from deepvoice3_pytorch_b200 import ops
    monkeypatch.setattr(ops, "tc_attention", True)
    return Spy(ops, monkeypatch)


def run(spy, name, mode, p, training=True):
    """One forward + backward of ops.attention_core on the case's inputs -> (results on CPU, mask M or None, calls)."""
    ops = spy.ops
    spy.mp.setattr(ops, "conv_math", mode)
    q, k, v, R1, R2 = A.inputs(name)
    mask = A.key_mask(name)
    qc, kc, vc = [t.cuda().requires_grad_(True) for t in (q, k, v)]
    ops.rng.manual_seed(SEED, qc.device)
    ops.rng.start_forward()
    spy.clear()
    out, probs = ops.attention_core(qc, kc, vc, None if mask is None else mask.cuda(), p, training)
    ((out * R1.cuda()).sum() + (probs * R2.cuda()).sum()).backward()
    torch.cuda.synchronize()
    calls = list(spy.calls)
    assert len(spy.draws) == 1
    p_eff, seed_t, salt = spy.draws[0]
    M = None
    if p_eff > 0:
        assert p_eff == p and salt != 0
        M = rebuild_mask(spy, probs.shape, p_eff, seed_t, salt)
    res = {"out": out.detach().cpu(), "probs": probs.detach().cpu(), "dq": qc.grad.cpu(), "dk": kc.grad.cpu(),
           "dv": vc.grad.cpu()}
    return res, M, calls


def check_path(name, mode, calls):
    path = A.path_of(name, mode)
    if path == "tc":
        assert "dv3_tc_attn_fwd" in calls and "dv3_tc_attn_bwd" in calls, calls
        assert "dv3_softmax_fwd" not in calls and "dv3_bgemm" not in calls, calls
    else:
        assert not any(c.startswith("dv3_tc_attn") for c in calls), calls
        assert {"dv3_bgemm", "dv3_softmax_fwd", "dv3_softmax_bwd"} <= set(calls), calls
    return path


def errors(name, res, M):
    q, k, v, R1, R2 = A.inputs(name)
    ref = A.reference(q, k, v, A.key_mask(name), M, R1, R2)
    return {t: A.relerr(res[t], ref[t]) for t in A.TENSORS}


@pytest.mark.parametrize("mode", ["tc", "fp32"])
@pytest.mark.parametrize("name", list(A.CASES))
def test_attention_core_vs_float64(name, mode, spy):
    p = A.CASES[name][5]
    res0, M0, calls = run(spy, name, mode, 0.0)
    path = check_path(name, mode, calls)
    assert M0 is None
    err0 = errors(name, res0, None)
    for t in A.TENSORS:
        assert err0[t] <= A.bound(name, path, t), (t, err0[t], A.bound(name, path, t))
    if p == 0.0:
        return
    res, M, calls = run(spy, name, mode, p)
    assert check_path(name, mode, calls) == path
    err = errors(name, res, M)
    for t in A.TENSORS:
        b = A.bound(name, path, t)
        assert err[t] <= b, ("p=%g" % p, t, err[t], b)
        assert err[t] <= A.DROP_RATIO * err0[t] + A.DROP_FLOOR * b, ("p=%g" % p, t, err[t], err0[t])


@pytest.mark.parametrize("mode", ["tc", "fp32"])
@pytest.mark.parametrize("name", ["b3_e144_td127_ts100", "simt_b3_e256_td128_ts200"])
def test_eval_ignores_dropout(name, mode, spy):
    """training=False with p > 0 computes exactly what p = 0 computes, and draws no dropout salt."""
    a, _, _ = run(spy, name, mode, 0.0)
    b, M, _ = run(spy, name, mode, 0.5, training=False)
    assert M is None and spy.draws[0] == (0.0, None, 0)
    for t in A.TENSORS:
        assert torch.equal(a[t], b[t]), t


@pytest.mark.parametrize("name", ["bench_b16_e256_td200_ts128", "b3_e144_td127_ts100"])
def test_tc_attention_is_deterministic(name, spy):
    """No atomics in the tensor-core attention: two identical calls agree bit for bit, forward and backward."""
    a, Ma, calls = run(spy, name, "tc", A.CASES[name][5])
    assert "dv3_tc_attn_fwd" in calls
    b, Mb, _ = run(spy, name, "tc", A.CASES[name][5])
    assert torch.equal(Ma, Mb)
    for t in A.TENSORS:
        assert torch.equal(a[t], b[t]), t


def _seed(dev):
    return torch.tensor([0x1234ABCD5678], dtype=torch.int64, device=dev)


def test_tc_attn_bwd_null_dprobs(spy):
    """dv3_tc_attn_bwd with dprobs = null (autograd always passes a tensor): the same bits as a zero dprobs, and the
    float64 gradient of <out, R1> alone."""
    ops = spy.ops
    name, p, salt = "b3_e144_td127_ts100", 0.5, 11
    B, E, Td, Ts = A.CASES[name][:4]
    q, k, v, R1, _ = A.inputs(name)
    mask = A.key_mask(name)
    qc, kc, vc, dout = [t.cuda() for t in (q, k, v, R1)]
    mc = mask.to(torch.uint8).cuda()
    seed_t = _seed(qc.device)
    sc = A.scale_of(Ts)
    probs = torch.empty(B, Td, Ts, device="cuda")
    out = torch.empty(B, E, Td, device="cuda")
    P = ops._p
    spy.raw_call("dv3_tc_attn_fwd", P(qc), P(kc), P(vc), P(mc), P(probs), P(out), B, E, Td, Ts, sc, p, P(seed_t), salt,
                 ops._stream())
    grads = []
    for dprobs in (None, torch.zeros(B, Td, Ts, device="cuda")):
        ds = torch.empty(B, Td, Ts, device="cuda")
        dq, dk, dv = torch.empty_like(qc), torch.empty_like(kc), torch.empty_like(vc)
        spy.raw_call("dv3_tc_attn_bwd", P(dout), P(qc), P(kc), P(vc), P(probs), P(dprobs), P(ds), P(dq), P(dk), P(dv),
                     B, E, Td, Ts, sc, p, P(seed_t), salt, ops._stream())
        grads.append({"dq": dq.cpu(), "dk": dk.cpu(), "dv": dv.cpu(), "ds": ds.cpu()})
    for t in grads[0]:
        assert torch.equal(grads[0][t], grads[1][t]), t
    M = rebuild_mask(spy, (B, Td, Ts), p, seed_t, salt)
    ref = A.reference(q, k, v, mask, M, R1, torch.zeros(B, Td, Ts))
    res = {"out": out.cpu(), "probs": probs.cpu(), **grads[0]}
    for t in A.TENSORS:
        assert A.relerr(res[t], ref[t]) <= A.bound(name, "tc", t), t


def test_softmax_bwd_null_dprobs(spy):
    """dv3_softmax_bwd (SIMT path) with dprobs_ext = null: the same bits as a zero tensor, and dS = P * (g - <g, P>)
    with g = dPd * M in float64."""
    ops = spy.ops
    name, p, salt = "simt_b3_e256_td128_ts200", 0.5, 5
    B, E, Td, Ts = A.CASES[name][:4]
    q, k, _, _, _ = A.inputs(name)
    mask = A.key_mask(name)
    S = torch.bmm(q.double().transpose(1, 2), k.double()).float()
    dpd = torch.randn(B, Td, Ts, generator=torch.Generator().manual_seed(3))
    Sc, dpdc, mc = S.cuda(), dpd.cuda(), mask.to(torch.uint8).cuda()
    seed_t = _seed(Sc.device)
    P = ops._p
    probs, pd = torch.empty_like(Sc), torch.empty_like(Sc)
    spy.raw_call("dv3_softmax_fwd", P(Sc), P(mc), P(probs), P(pd), B * Td, Ts, Td, p, P(seed_t), salt, ops._stream())
    dss = []
    for dprobs in (None, torch.zeros_like(Sc)):
        ds = torch.empty_like(Sc)
        spy.raw_call("dv3_softmax_bwd", P(probs), P(dpdc), P(dprobs), P(ds), B * Td, Ts, p, P(seed_t), salt,
                     ops._stream())
        dss.append(ds.cpu())
    assert torch.equal(dss[0], dss[1])
    M = rebuild_mask(spy, (B, Td, Ts), p, seed_t, salt)
    Pr = torch.softmax(S.double().masked_fill(mask[:, None, :], -math.inf), dim=-1)
    g = dpd.double() * M.double()
    ds_ref = Pr * (g - (g * Pr).sum(-1, keepdim=True))
    assert A.relerr(probs.cpu(), Pr) <= A.bound(name, "fp32", "probs")
    assert A.relerr(pd.cpu(), Pr * M.double()) <= A.bound(name, "fp32", "probs")
    assert A.relerr(dss[0], ds_ref) <= A.bound(name, "fp32", "dq")


@pytest.mark.parametrize("mode,Ts", [("tc", 48), ("fp32", 48), ("tc", 160)])
def test_fully_masked_rows_are_nan(mode, Ts, spy):
    """An utterance whose keys are all masked has no softmax: both paths return NaN for its probabilities, context and
    dv, as the float64 reference does (softmax of a row of -inf), and NaN for its dq and dk, where the reference's
    masked_fill gives 0 (its loss is NaN either way).  The other utterances are unaffected."""
    ops = spy.ops
    spy.mp.setattr(ops, "conv_math", mode)
    B, E, Td = 2, 64, 40
    gen = torch.Generator().manual_seed(Ts)
    q, k = torch.randn(B, E, Td, generator=gen) * 0.2, torch.randn(B, E, Ts, generator=gen) * 0.2
    v = torch.randn(B, E, Ts, generator=gen)
    mask = torch.zeros(B, Ts, dtype=torch.bool)
    mask[0] = True
    mask[1, 33:] = True
    R1, R2 = torch.randn(B, E, Td, generator=gen), torch.randn(B, Td, Ts, generator=gen)
    qc, kc, vc = [t.cuda().requires_grad_(True) for t in (q, k, v)]
    ops.rng.manual_seed(SEED, qc.device)
    ops.rng.start_forward()
    spy.clear()
    out, probs = ops.attention_core(qc, kc, vc, mask.cuda(), 0.05, True)
    ((out * R1.cuda()).sum() + (probs * R2.cuda()).sum()).backward()
    tc_ran = "dv3_tc_attn_fwd" in spy.calls
    assert tc_ran == (mode == "tc" and Ts <= A.TC_MAX_TS)
    _, seed_t, salt = spy.draws[0]
    M = rebuild_mask(spy, (B, Td, Ts), 0.05, seed_t, salt)
    ref = A.reference(q, k, v, mask, M, R1, R2)
    res = {"out": out.detach().cpu(), "probs": probs.detach().cpu(), "dq": qc.grad.cpu(), "dk": kc.grad.cpu(),
           "dv": vc.grad.cpu()}
    path = "tc" if tc_ran else "fp32"
    for t in A.TENSORS:
        assert torch.isnan(res[t][0]).all(), (path, t)
        if t in ("dq", "dk"):          # the reference's masked_fill backward zeroes the gradient at every masked key
            assert torch.all(ref[t][0] == 0), t
        else:
            assert torch.isnan(ref[t][0]).all(), t
        assert torch.isfinite(res[t][1]).all(), (path, t)
        assert A.relerr(res[t][1], ref[t][1]) <= A.BOUNDS[(path, "align")][t], (path, t)
