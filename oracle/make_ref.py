#!/usr/bin/env python
"""TEST / BENCH INFRASTRUCTURE -- builds ``oracle/_ref``: a runnable copy of the UNMODIFIED reference.

    python oracle/make_ref.py            (build container only: needs /root/reference)

The reference is pure Python, so "building" it is: copy the package and the four top-level modules ``train.py``
imports (``train.py``, ``hparams.py``, ``lrschedule.py``, ``audio.py``), ``synthesis.py``, ``ljspeech.py`` and ``presets/`` from where they lie under
/root/reference into ``oracle/_ref/`` and generate ``deepvoice3_pytorch/version.py`` the way ``setup.py:33-39`` does.
``oracle/_ref/`` is git-ignored (no reference source enters the history) but NOT gpurun-ignored, so it travels to
the GPU box, where /root/reference does not exist.  Consumers (all test / bench side, never the product package):

* ``bench.py --impl reference``      the reference's own modules + losses + Adam on the host CPU (kind "reference")
* ``bench.py`` ``gpu_eager_baseline``  the same modules through PyTorch eager (cuDNN/cuBLAS) on the B200
* ``tests/golden/make_train_golden.py``  fixtures for the loss / collate functions of ``train.py``
* ``tests/golden/make_dropin_golden.py``  fixtures of ``train.py`` / ``synthesis.py`` / ``ljspeech.py`` run on the
                                          reference package, for ``tests/test_dropin.py``
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
FILES = ["train.py", "hparams.py", "lrschedule.py", "audio.py", "synthesis.py", "ljspeech.py"]


def build(ref="/root/reference", quiet=False):
    """-> path of oracle/_ref, or None when the reference tree is not present (GPU box: use what travelled)."""
    if not os.path.isdir(ref):
        return DST if os.path.isdir(os.path.join(DST, "deepvoice3_pytorch")) else None
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    os.makedirs(DST)
    shutil.copytree(os.path.join(ref, "deepvoice3_pytorch"), os.path.join(DST, "deepvoice3_pytorch"),
                    ignore=shutil.ignore_patterns("__pycache__"))
    with open(os.path.join(DST, "deepvoice3_pytorch", "version.py"), "w") as f:
        f.write('__version__ = "0.1.1"\n')              # what setup.py:33-39 generates at install time
    for name in FILES:
        shutil.copy(os.path.join(ref, name), os.path.join(DST, name))
    shutil.copytree(os.path.join(ref, "presets"), os.path.join(DST, "presets"))
    fixture = os.path.join(ref, "tests", "data", "ljspeech-mel-00001.npy")
    if os.path.exists(fixture):
        shutil.copy(fixture, os.path.join(DST, "ljspeech-mel-00001.npy"))
    if not quiet:
        n = sum(len(fs) for _, _, fs in os.walk(DST))
        print("oracle/_ref: %d files copied from %s" % (n, ref))
    return DST


def path():
    """oracle/_ref if it has been built (here or shipped), else None."""
    return DST if os.path.isdir(os.path.join(DST, "deepvoice3_pytorch")) else None


if __name__ == "__main__":
    sys.exit(0 if build() else 1)
