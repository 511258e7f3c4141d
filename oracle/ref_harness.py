"""TEST / BENCH INFRASTRUCTURE -- loads the reference's own ``train.py`` (from ``oracle/_ref``) UNCHANGED,
on top of either the reference package or ``deepvoice3_pytorch_b200``.

``train.py`` imports a number of packages that are not installed here and that the training hot path never touches
(docopt: CLI; nnmnkwii: file datasets; tensorboardX / matplotlib / librosa.display: logging and plots; nltk: the
CMU dictionary of the English text frontend; lws / librosa: audio.py).  They are replaced by empty stand-ins in
``sys.modules`` -- calling into one of them raises -- and ``np.int`` (removed in numpy 1.24, used by
``train.py:319,335``) is restored as an alias of ``int``.  Nothing of the reference is edited.

    tr = load_train("b200")        # reference train.py, with `from deepvoice3_pytorch import builder` -> our package
    tr = load_train("reference")   # the same file on the reference package
"""
import importlib.util
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
N_VOCAB = 149          # len(symbols) of the reference's English frontend (frontend/text/symbols.py)


def ref_root():
    """oracle/_ref when it has been built (oracle/make_ref.py), else None."""
    from oracle import make_ref
    return make_ref.path()


class _Missing(types.ModuleType):
    """Stand-in for an uninstalled dependency: importable, but any use raises."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        raise ImportError("%s.%s: this dependency of the reference is not installed (stubbed by oracle/ref_harness.py)"
                          % (self.__name__, name))


class ScalarLog:
    """tensorboardX.SummaryWriter stand-in that keeps the scalars train.py logs (train.py:761-776)."""

    def __init__(self, *a, **kw):
        self.scalars = {}

    def add_scalar(self, tag, value, step=None):
        self.scalars.setdefault(tag, []).append((step, float(value)))

    def add_image(self, *a, **kw):
        pass

    def add_audio(self, *a, **kw):
        pass

    def close(self):
        pass


def install_stubs():
    if not hasattr(np, "int"):
        np.int = int                                      # train.py:319,335 (numpy < 1.24 spelling)

    def mod(name, **attrs):
        if name in sys.modules and not isinstance(sys.modules[name], _Missing):
            return sys.modules[name]
        m = _Missing(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    mod("docopt", docopt=lambda *a, **kw: {})
    nn_ = mod("nnmnkwii")
    nn_.__path__ = []
    nn_.datasets = mod("nnmnkwii.datasets", FileSourceDataset=object, FileDataSource=object)
    nn_.preprocessing = mod("nnmnkwii.preprocessing")
    mod("tensorboardX", SummaryWriter=ScalarLog)
    mpl = mod("matplotlib", use=lambda *a, **kw: None)
    mpl.__path__ = []
    mpl.pyplot = mod("matplotlib.pyplot")
    mpl.cm = mod("matplotlib.cm")
    lib = mod("librosa")
    lib.__path__ = []
    lib.display = mod("librosa.display")
    lib.filters = mod("librosa.filters")
    lib.core = mod("librosa.core")
    mod("lws")
    mod("unidecode", unidecode=lambda s: s)               # frontend/text/cleaners.py, numbers.py (text path only)
    mod("inflect", engine=lambda: None)
    nltk = mod("nltk")
    nltk.corpus = types.SimpleNamespace(cmudict=types.SimpleNamespace(dict=lambda: {}))


def _load_file(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


_PKG_KEYS = ("deepvoice3_pytorch",)


def _drop_package():
    for k in [k for k in sys.modules if k == "deepvoice3_pytorch" or k.startswith("deepvoice3_pytorch.")]:
        del sys.modules[k]


def bind_package(which, root=None):
    """Make ``import deepvoice3_pytorch`` resolve to the reference package ("reference") or to
    ``deepvoice3_pytorch_b200`` ("b200": what a user does by installing this package under the reference's name)."""
    root = root or ref_root()
    install_stubs()
    _drop_package()
    if which == "reference":
        if root not in sys.path:
            sys.path.insert(0, root)
        import deepvoice3_pytorch                      # noqa: F401  (frontend pulls the nltk stand-in)
        return sys.modules["deepvoice3_pytorch"]
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import deepvoice3_pytorch_b200 as pkg
    from deepvoice3_pytorch_b200 import builder
    sys.modules["deepvoice3_pytorch"] = pkg
    sys.modules["deepvoice3_pytorch.builder"] = builder
    fe = types.ModuleType("deepvoice3_pytorch.frontend")   # train.py only reads frontend.<lang>.n_vocab (:816)
    fe.en = types.SimpleNamespace(n_vocab=N_VOCAB)
    sys.modules["deepvoice3_pytorch.frontend"] = fe
    pkg.frontend = fe
    # hparams.py needs the vendored HParams class (deepvoice3_pytorch/tfcompat/hparam.py): plain Python, loaded as is
    tf = types.ModuleType("deepvoice3_pytorch.tfcompat")
    tf.__path__ = [os.path.join(root, "deepvoice3_pytorch", "tfcompat")]
    sys.modules["deepvoice3_pytorch.tfcompat"] = tf
    _load_file("deepvoice3_pytorch.tfcompat.hparam", os.path.join(root, "deepvoice3_pytorch", "tfcompat", "hparam.py"))
    return pkg


def load_train(which="b200", root=None):
    """Execute the reference's train.py (module level only: no ``__main__``) bound to the chosen package.
    Returns the module; ``.hparams`` is the shared reference HParams object."""
    root = root or ref_root()
    if root is None:
        raise RuntimeError("no reference tree: run `python oracle/make_ref.py` in the build container")
    pkg = bind_package(which, root)
    if root not in sys.path:
        sys.path.insert(0, root)                           # hparams, lrschedule, audio: train.py's siblings
    for k in ("hparams", "audio", "lrschedule"):
        sys.modules.pop(k, None)
    m = _load_file("dv3_ref_train_" + which, os.path.join(root, "train.py"))
    fe = sys.modules["deepvoice3_pytorch.frontend"]
    m._frontend = getattr(fe, "en")                       # train.py:950 (`getattr(frontend, hparams.frontend)`)
    m._package = pkg
    return m


class CharFrontend:
    """Stand-in for ``deepvoice3_pytorch.frontend.en`` (nltk / CMU dictionary are not installed): one id per
    character, ids in [2, N_VOCAB) like the reference's symbol table, 1 = end of sentence."""
    n_vocab = N_VOCAB

    @staticmethod
    def text_to_sequence(text, p=0.0):
        return [2 + (ord(c) * 7) % (N_VOCAB - 2) for c in text] + [1]


def load_synthesis(which="b200", audio_module=None, root=None):
    """Execute the reference's synthesis.py (module level only) bound to the chosen package.  ``audio_module`` is what
    its ``import audio`` resolves to: this package's ``audio`` for "b200"; for "reference" a shim must be passed (the
    reference's audio.py needs the uninstalled ``lws`` for the inverse path).  ``tts()`` is then callable unchanged."""
    root = root or ref_root()
    if root is None:
        raise RuntimeError("no reference tree: run `python oracle/make_ref.py` in the build container")
    pkg = bind_package(which, root)
    if root not in sys.path:
        sys.path.insert(0, root)
    for k in ("hparams", "audio"):
        sys.modules.pop(k, None)
    if audio_module is not None:
        sys.modules["audio"] = audio_module
    m = _load_file("dv3_ref_synthesis_" + which, os.path.join(root, "synthesis.py"))
    m._frontend = CharFrontend
    m._package = pkg
    return m


def load_ljspeech(audio_module, root=None):
    """Execute the reference's ljspeech.py (the LJSpeech preprocessor: ``build_from_path`` / ``_process_utterance``)
    with ``import audio`` resolving to ``audio_module`` and ``hparams`` to the reference's own hparams.py."""
    root = root or ref_root()
    if root is None:
        raise RuntimeError("no reference tree: run `python oracle/make_ref.py` in the build container")
    bind_package("b200", root)                             # hparams.py needs the vendored tfcompat.hparam only
    if root not in sys.path:
        sys.path.insert(0, root)
    sys.modules.pop("hparams", None)
    sys.modules["audio"] = audio_module
    return _load_file("dv3_ref_ljspeech", os.path.join(root, "ljspeech.py"))


def apply_preset(tr, name, **overrides):
    """hparams.parse_json(presets/<name>.json) (train.py:936-939) + keyword overrides."""
    with open(os.path.join(ref_root(), "presets", name + ".json")) as f:
        tr.hparams.parse_json(f.read())
    for k, v in overrides.items():
        tr.hparams.set_hparam(k, v)
    return tr.hparams


def synthetic_utterances(n, seed=0, n_speakers=1, min_text=20, max_text=60, min_frames=80, max_frames=200,
                         linear_dim=513, mel_dim=80):
    """What ``PyTorchDataset.__getitem__`` (train.py:247-255) returns: (text ids, mel (T,80), linear (T,513)[, spk])."""
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        nt, nf = int(rng.randint(min_text, max_text + 1)), int(rng.randint(min_frames, max_frames + 1))
        item = (rng.randint(2, N_VOCAB, nt).astype(np.int64), rng.rand(nf, mel_dim).astype(np.float32),
                rng.rand(nf, linear_dim).astype(np.float32))
        if n_speakers > 1:
            item = item + (int(rng.randint(0, n_speakers)),)
        out.append(item)
    return out
