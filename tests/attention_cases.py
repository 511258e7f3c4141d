"""Shared by tests/test_gpu_attention_core.py and tests/test_attention_tolerance.py: the attention-core cases, their
inputs, a float64 reference, an emulation of the tensor-core arithmetic and the error bounds the GPU test applies.

The attention core (ops.attention_core, reference deepvoice3.py:143-171):
    S = q^T k (no 1/sqrt(d)) -> padded keys -inf -> P = softmax over keys -> Pd = P * M -> out = scale * v Pd^T
with scale = Ts * sqrt(1/Ts) and M the dropout mask (0 or 1/(1-p)).  The loss the tests differentiate is
<out, R1> + <P, R2>.

The tensor-core kernels (csrc/tc_attn.cu) compute every contraction as hi*hi' + hi*lo' + lo*hi' with hi = bf16(x) and
lo = bf16(x - hi).  emulate() runs the same forward and backward in float64 with that product ("split") or with
hi*hi' only ("hi"); the bounds below sit between the two, so a kernel that loses a cross term fails and a correct one
passes with margin.  test_attention_tolerance.py checks that for every case."""
import math

import numpy as np
import torch

import golden_util as G

TENSORS = ("out", "probs", "dq", "dk", "dv")
WINDOW_LAST_ATTENDED, WINDOW_BACKWARD, WINDOW_AHEAD = 31, 1, 3     # AttentionLayer.forward defaults; crosses key 32
RAGGED_LENGTHS = (95, 33, 32, 31, 1)

# name: (B, E, Td, Ts, mask, p, score_std, with_R2).  Curated so that every kernel boundary is hit at least once:
# E not a multiple of 64 (partial K chunks) and in (128, 256) (a partial second CTA of attn_cols_kernel); Ts at the
# 32 / 64 / 128 edges of the ballot words and key slabs; Td odd / not a multiple of 4 / several CTAs; Ts > 128 takes
# the SIMT kernels (dv3_bgemm + dv3_softmax_*) even in tensor-core mode.
CASES = {
    "b1_e16_td1_ts1":          (1, 16, 1, 1, "none", 0.0, 3.0, True),
    "b3_e16_td5_ts7":          (3, 16, 5, 7, "ragged", 0.5, 3.0, True),
    "b1_e16_td803_ts7":        (1, 16, 803, 7, "none", 0.05, 3.0, True),
    "b3_e48_td127_ts31":       (3, 48, 127, 31, "ragged", 0.05, 3.0, True),
    "b3_e48_td128_ts32_noR2":  (3, 48, 128, 32, "none", 0.5, 3.0, False),
    "b3_e80_td129_ts33":       (3, 80, 129, 33, "ragged", 0.05, 3.0, True),
    "b3_e80_td5_ts31_window":  (3, 80, 5, 31, "window", 0.0, 3.0, True),
    "b1_e80_td200_ts64_window": (1, 80, 200, 64, "window", 0.5, 3.0, True),
    "b3_e128_td5_ts65":        (3, 128, 5, 65, "ragged", 0.05, 3.0, True),
    "b1_e128_td129_ts32":      (1, 128, 129, 32, "ragged", 0.5, 3.0, True),
    "b3_e144_td127_ts100":     (3, 144, 127, 100, "ragged", 0.5, 3.0, True),
    "b16_e144_td129_ts127_noR2": (16, 144, 129, 127, "ragged", 0.05, 3.0, False),
    "b3_e144_td1_ts128":       (3, 144, 1, 128, "none", 0.5, 3.0, True),
    "b3_e256_td128_ts33_noR2": (3, 256, 128, 33, "none", 0.5, 3.0, False),
    "b3_e256_td129_ts100_window": (3, 256, 129, 100, "window", 0.05, 3.0, True),
    "b3_e256_td803_ts128":     (3, 256, 803, 128, "ragged", 0.05, 3.0, True),
    "b16_e48_td127_ts65":      (16, 48, 127, 65, "ragged", 0.0, 3.0, True),
    "b3_e48_td200_ts64_onehot": (3, 48, 200, 64, "none", 0.05, 30.0, True),
    "b3_e128_td200_ts100_onehot": (3, 128, 200, 100, "ragged", 0.5, 30.0, True),
    "bench_b16_e256_td200_ts128": (16, 256, 200, 128, "ragged", 0.05, 3.0, True),
    "nyanko_b16_e128_td200_ts128": (16, 128, 200, 128, "ragged", 0.05, 3.0, True),
    # Ts > 128: the SIMT kernels in both modes
    "simt_b3_e128_td200_ts129": (3, 128, 200, 129, "ragged", 0.05, 3.0, True),
    "simt_b3_e144_td5_ts129_window": (3, 144, 5, 129, "window", 0.0, 3.0, False),
    "simt_b3_e256_td128_ts200": (3, 256, 128, 200, "ragged", 0.5, 3.0, True),
    "simt_b1_e80_td127_ts511": (1, 80, 127, 511, "ragged", 0.05, 3.0, True),
    "simt_b3_e48_td129_ts200_onehot": (3, 48, 129, 200, "none", 0.05, 30.0, True),
}

TC_MAX_TS = 128        # dv3_tc_attn_supported: longer key axes run on the SIMT kernels


def regime(name):
    return "onehot" if CASES[name][6] > 10 else "align"


# Relative-L2 bounds per tensor, by arithmetic and score regime ("align": score std ~3 like trained alignments;
# "onehot": std ~30, near one-hot rows).  "tc": tensor-core kernels; "fp32": the exact-fp32 SIMT kernels (fp32 mode,
# and Ts > 128 in tc mode).  Calibrated by test_attention_tolerance.py; the emulated errors behind each entry are
# printed by `python tests/test_attention_tolerance.py`.
BOUNDS = {
    ("tc", "align"):    {"out": 1e-4, "probs": 1e-4, "dq": 2e-4, "dk": 2e-4, "dv": 1e-4},
    ("tc", "onehot"):   {"out": 3e-4, "probs": 3e-4, "dq": 1e-3, "dk": 1e-3, "dv": 3e-4},
    ("fp32", "align"):  {"out": 3e-5, "probs": 3e-5, "dq": 3e-5, "dk": 3e-5, "dv": 3e-5},
    ("fp32", "onehot"): {"out": 5e-5, "probs": 5e-5, "dq": 2e-4, "dk": 2e-4, "dv": 5e-5},
}

# err(p > 0) <= DROP_RATIO * err(p = 0) + DROP_FLOOR * bound: dropout rescales kept terms by 1/(1-p) and zeroes the
# rest, which leaves the relative error of a correct kernel about where it is without dropout, while a mask
# regenerated at a wrong index changes the result by O(1).
DROP_RATIO, DROP_FLOOR = 2.0, 0.25


def path_of(name, mode):
    """Which kernels a case runs on in ops.conv_math mode ``mode``."""
    return "tc" if mode == "tc" and CASES[name][3] <= TC_MAX_TS else "fp32"


def bound(name, path, tensor):
    return BOUNDS[(path, regime(name))][tensor]


def key_mask(name):
    """(B, Ts) bool, True = excluded key, or None."""
    B, E, Td, Ts, kind = CASES[name][:5]
    s = torch.arange(Ts)
    if kind == "none":
        return None
    if kind == "ragged":
        lengths = [Ts] + [n for n in RAGGED_LENGTHS if n < Ts]
        lengths = torch.tensor([lengths[b % len(lengths)] for b in range(B)])
        return s[None, :] >= lengths[:, None]
    # deepvoice3.AttentionLayer.forward with last_attended: keys outside [la - backward, la + ahead) are excluded
    lo, hi = WINDOW_LAST_ATTENDED - WINDOW_BACKWARD, WINDOW_LAST_ATTENDED + WINDOW_AHEAD
    win = torch.zeros(Ts, dtype=torch.bool)
    if lo > 0:
        win |= s < lo
    if hi < Ts:
        win |= s >= hi
    return win[None, :].expand(B, Ts).contiguous()


def inputs(name):
    """float32 CPU tensors q (B,E,Td), k, v (B,E,Ts), R1 (B,E,Td), R2 (B,Td,Ts) (zeros when the case has no R2).
    q and k ~ N(0, sigma^2) with sigma^2 sqrt(E) = score_std."""
    B, E, Td, Ts, _, _, std, with_r2 = CASES[name]
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    sig = math.sqrt(std / math.sqrt(E))
    q = torch.randn(B, E, Td, generator=gen) * sig
    k = torch.randn(B, E, Ts, generator=gen) * sig
    v = torch.randn(B, E, Ts, generator=gen)
    R1 = G.loss_weights((B, E, Td), 0)
    R2 = G.loss_weights((B, Td, Ts), 1) if with_r2 else torch.zeros(B, Td, Ts)
    return q, k, v, R1, R2


def scale_of(Ts):
    return Ts * math.sqrt(1.0 / Ts)


def reference(q, k, v, mask, M, R1, R2, dtype=torch.float64):
    """Autograd reference in ``dtype`` on the CPU -> {out, probs, dq, dk, dv}.  M: (B,Td,Ts) dropout mask or None."""
    q, k, v = [t.detach().to(dtype).requires_grad_(True) for t in (q, k, v)]
    S = torch.bmm(q.transpose(1, 2), k)
    if mask is not None:
        S = S.masked_fill(mask[:, None, :], -math.inf)
    P = torch.softmax(S, dim=-1)
    Pd = P if M is None else P * M.to(dtype)
    out = scale_of(k.shape[2]) * torch.bmm(v, Pd.transpose(1, 2))
    loss = (out * R1.to(dtype)).sum() + (P * R2.to(dtype)).sum()
    loss.backward()
    return {"out": out.detach(), "probs": P.detach(), "dq": q.grad, "dk": k.grad, "dv": v.grad}


def _split(x):
    x32 = x.float()
    hi = x32.to(torch.bfloat16).float()
    lo = (x32 - hi).to(torch.bfloat16).float()
    return hi.double(), lo.double()


def _mm(a, b, arith):
    """batched a @ b in float64 with the operands split the way the tensor-core kernels split them."""
    ah, al = _split(a)
    bh, bl = _split(b)
    d = torch.bmm(ah, bh)
    if arith == "split":
        d = d + torch.bmm(ah, bl) + torch.bmm(al, bh)
    return d


def emulate(q, k, v, mask, M, R1, R2, arith):
    """The forward and backward contractions of csrc/tc_attn.cu with product ``arith`` ("split" | "hi"), everything
    else in float64 -> {out, probs, dq, dk, dv}."""
    q, k, v, R1, R2 = [t.double() for t in (q, k, v, R1, R2)]
    M = torch.ones(1, dtype=torch.float64) if M is None else M.double()
    sc = scale_of(k.shape[2])
    S = _mm(q.transpose(1, 2), k, arith)                            # attn_rows_kernel<0>, GEMM 1
    if mask is not None:
        S = S.masked_fill(mask[:, None, :], -math.inf)
    P = torch.softmax(S, dim=-1)
    Pd = P * M
    out = sc * _mm(Pd, v.transpose(1, 2), arith).transpose(1, 2)   # GEMM 2
    dPd = sc * _mm(R1.transpose(1, 2), v, arith)                    # attn_rows_kernel<1>, GEMM 1
    g = dPd * M + R2
    dS = P * (g - (g * P).sum(-1, keepdim=True))
    dq = _mm(dS, k.transpose(1, 2), arith).transpose(1, 2)          # GEMM 2
    dv = sc * _mm(R1, Pd, arith)                                    # attn_cols_kernel
    dk = _mm(q, dS, arith)
    return {"out": out, "probs": P, "dq": dq, "dk": dk, "dv": dv}


def relerr(x, ref):
    """||x - ref|| / ||ref|| (0 when both vanish, inf when only ref does)."""
    x, ref = x.double().cpu(), ref.double().cpu()
    num, den = float(torch.linalg.vector_norm(x - ref)), float(torch.linalg.vector_norm(ref))
    if den == 0.0:
        return 0.0 if num == 0.0 else math.inf
    return num / den


def cpu_dropout_mask(name, p):
    """A mask with the kernels' keep rate and scale from torch's RNG (the tolerance calibration has no GPU)."""
    B, E, Td, Ts = CASES[name][:4]
    if p == 0.0:
        return None
    gen = torch.Generator().manual_seed(7)
    return (torch.rand(B, Td, Ts, generator=gen) >= p).float() / (1.0 - p)
