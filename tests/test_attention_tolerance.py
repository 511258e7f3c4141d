"""Calibration of the attention-core error bounds (attention_cases.BOUNDS) that test_gpu_attention_core.py applies.

For every case: the tensor-core bound of each tensor is at least 4x the error of a float64 emulation of the kernels'
split-bf16 products (hi*hi' + hi*lo' + lo*hi') and at most 1/4 of the error of the same emulation with hi*hi' only,
so a kernel that drops a cross term fails it and a correct one passes with margin.  The exact-fp32 bound is at least
4x the error of a CPU float32 run of the same ops and likewise at most 1/4 of the hi-only error.  Errors are relative
L2 against the float64 reference.  CPU only.

    python tests/test_attention_tolerance.py     prints the emulated errors behind every bound"""
import functools

import pytest
import torch

import attention_cases as A

LOW, HIGH = 4.0, 0.25
SENSITIVE = 1e-9       # a tensor whose hi-only error is below this does not depend on operand precision (Ts = 1 rows)


@functools.lru_cache(maxsize=None)
def measured(name, p):
    """-> {arith: {tensor: relerr vs float64}} for arith in split / hi / fp32."""
    q, k, v, R1, R2 = A.inputs(name)
    mask, M = A.key_mask(name), A.cpu_dropout_mask(name, p)
    ref = A.reference(q, k, v, mask, M, R1, R2)
    runs = {"split": A.emulate(q, k, v, mask, M, R1, R2, "split"),
            "hi": A.emulate(q, k, v, mask, M, R1, R2, "hi"),
            "fp32": A.reference(q, k, v, mask, M, R1, R2, dtype=torch.float32)}
    return {a: {t: A.relerr(r[t], ref[t]) for t in A.TENSORS} for a, r in runs.items()}


def _ps(name):
    p = A.CASES[name][5]
    return (0.0, p) if p > 0 else (0.0,)


def test_emulated_backward_is_the_reference_gradient():
    """emulate() writes the backward out by hand, as the kernels compute it; with exact products it must be the
    autograd gradient, or the calibration would measure something else."""
    name = "b3_e80_td129_ts33"
    q, k, v, R1, R2 = A.inputs(name)
    mask, M = A.key_mask(name), A.cpu_dropout_mask(name, 0.5)
    ref = A.reference(q, k, v, mask, M, R1, R2)
    orig = A._split
    try:
        A._split = lambda x: (x.double(), torch.zeros_like(x, dtype=torch.float64))
        exact = A.emulate(q, k, v, mask, M, R1, R2, "split")
    finally:
        A._split = orig
    for t in A.TENSORS:
        assert A.relerr(exact[t], ref[t]) < 1e-12, t


@pytest.mark.parametrize("name", list(A.CASES))
def test_bounds_between_split_and_hi_only(name):
    for p in _ps(name):
        m = measured(name, p)
        for path, lower in (("tc", "split"), ("fp32", "fp32")):
            for t in A.TENSORS:
                b = A.bound(name, path, t)
                assert b >= LOW * m[lower][t], (name, p, path, t, b, m[lower][t])
                if m["hi"][t] > SENSITIVE:
                    assert b <= HIGH * m["hi"][t], (name, p, path, t, b, m["hi"][t])


@pytest.mark.parametrize("name", [n for n in A.CASES if A.CASES[n][5] > 0])
def test_dropout_keeps_the_error_scale(name):
    """The p>0 vs p=0 check of the GPU test holds for the emulated kernels: dropout does not inflate the error."""
    p = A.CASES[name][5]
    for path, arith in (("tc", "split"), ("fp32", "fp32")):
        e0, e1 = measured(name, 0.0)[arith], measured(name, p)[arith]
        for t in A.TENSORS:
            assert e1[t] <= A.DROP_RATIO * e0[t] + A.DROP_FLOOR * A.bound(name, path, t), (name, path, t, e0[t], e1[t])


if __name__ == "__main__":
    for (path, reg), row in A.BOUNDS.items():
        names = [n for n in A.CASES if A.regime(n) == reg]
        lower = "split" if path == "tc" else "fp32"
        print("%s / %s" % (path, reg))
        for t in A.TENSORS:
            lo = max(measured(n, p)[lower][t] for n in names for p in _ps(n))
            hi = min(measured(n, p)["hi"][t] for n in names for p in _ps(n) if measured(n, p)["hi"][t] > SENSITIVE)
            print("  %-5s bound %.1e   max %s error %.1e   min hi-only error %.1e" % (t, row[t], lower, lo, hi))
