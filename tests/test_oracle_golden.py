"""CPU: the oracle restatement (oracle/) against the golden vectors produced by the live reference.
This is what "parity pinned" means for the model path (DESIGN.md section c)."""
import numpy as np
import pytest
import torch

from oracle import dv3_oracle as O
from oracle.specs import spec_from_builder
import golden_util as G

RTOL, ATOL = 1e-4, 1e-5      # oracle vs reference on CPU: same ATen kernels, tiny reassociation only


def close(a, b, rtol=RTOL, atol=ATOL):
    a = a.detach().numpy() if torch.is_tensor(a) else a
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def _grads(outs, leaves):
    loss = sum((o * G.loss_weights(o.shape, i)).sum() for i, o in enumerate(outs))
    return torch.autograd.grad(loss, leaves, allow_unused=True)


def _leaf_sd(case):
    sd = G.tensors(case["sd"])
    for k, v in sd.items():
        if v.is_floating_point():
            v.requires_grad_(True)
    return sd


def _check_case(case, outs, sd, inputs):
    for i, o in enumerate(outs):
        close(o, case["out"][str(i)])
    names = [k for k in case["gsd"]]
    leaves = [sd[k] for k in names] + [inputs[k] for k in case.get("gin", {})]
    grads = _grads(outs, leaves)
    for k, g in zip(names + list(case.get("gin", {})), grads):
        ref = case["gsd"][k] if k in case["gsd"] else case["gin"][k]
        # fp32 gradient sums carry rounding error in proportion to the tensor's largest entries, and its size depends
        # on the CPU's kernels: small entries of a large-valued weight gradient get an absolute allowance of 1e-5 of
        # that scale on top of 2e-4
        close(g, ref, rtol=1e-3, atol=2e-4 + 1e-5 * float(np.abs(ref).max()))


BLOCKS = G.load("blocks.npz")


@pytest.mark.parametrize("name", [n for n in BLOCKS if n.startswith("glu")])
def test_conv1d_glu(name):
    case = BLOCKS[name]
    sd = _leaf_sd(case)
    ins = G.tensors(case["in"])
    for v in ins.values():
        v.requires_grad_(True)
    m = {k: G.meta_scalar(case, k) for k in ("k", "d", "causal", "residual")}
    sdp = {"m." + k: v for k, v in sd.items()}
    y = O.conv1d_glu(sdp, "m", ins["x"], m["k"], m["d"], bool(m["causal"]), bool(m["residual"]),
                     ins.get("spk"))
    _check_case(case, (y,), sd, ins)


@pytest.mark.parametrize("name", [n for n in BLOCKS if n.startswith("hw")])
def test_highway(name):
    case = BLOCKS[name]
    sd = _leaf_sd(case)
    ins = G.tensors(case["in"])
    ins["x"].requires_grad_(True)
    m = {k: G.meta_scalar(case, k) for k in ("k", "d", "causal")}
    y = O.highway_conv1d({"m." + k: v for k, v in sd.items()}, "m", ins["x"], m["k"], m["d"],
                         bool(m["causal"]))
    _check_case(case, (y,), sd, ins)


@pytest.mark.parametrize("name,fn", [("conv1x1_0", "conv"), ("conv1x1_1", "conv"), ("convT", "convT"),
                                     ("linear", "linear")])
def test_weightnormed_leaf(name, fn):
    case = BLOCKS[name]
    sd = _leaf_sd(case)
    ins = G.tensors(case["in"])
    ins["x"].requires_grad_(True)
    sdp = {"m." + k: v for k, v in sd.items()}
    y = {"conv": lambda: O.conv1d(sdp, "m", ins["x"]),
         "convT": lambda: O.conv_transpose1d(sdp, "m", ins["x"]),
         "linear": lambda: O.linear(sdp, "m", ins["x"])}[fn]()
    _check_case(case, (y,), sd, ins)


@pytest.mark.parametrize("name", [n for n in BLOCKS if n.startswith("attn")])
def test_attention(name):
    case = BLOCKS[name]
    sd = _leaf_sd(case)
    ins = G.tensors(case["in"])
    for v in ins.values():
        v.requires_grad_(True)
    lengths = case["meta"]["lengths"]
    mask = O.memory_mask(lengths, ins["keys"].size(-1)) if lengths.size else None
    out, probs = O.attention_layer({"m." + k: v for k, v in sd.items()}, "m", ins["query"],
                                   ins["keys"], ins["values"], mask)
    _check_case(case, (out, probs), sd, ins)


@pytest.mark.parametrize("name", [n for n in BLOCKS if n.startswith("sin")])
def test_sinusoidal(name):
    case = BLOCKS[name]
    x = torch.from_numpy(case["in"]["x"])
    w = case["meta"]["w"]
    if name == "sin_batch":
        table = torch.from_numpy(case["sd"]["weight"])
        out = O.sinusoidal_encoding(table, x, torch.from_numpy(w))
    else:
        w = float(w)
        n, d = case["out"]["table"].shape
        table = O.position_table(n, d, 1.0, sinusoidal=False)
        out = O.sinusoidal_encoding(table, x, w)
        # position_encoding_init(rate=w) is the float64-argument table (modules.py:10-24)
        close(O.position_table(n, d, w, sinusoidal=True), case["out"]["table"], rtol=0, atol=0)
    close(out, case["out"]["0"], rtol=1e-6, atol=1e-6)


def test_conv_ramp_known_answer():
    """reference tests/test_conv.py:10-63 known-answer: exact integers."""
    ramp = G.load("conv_ramp.npz")
    for name, case in ramp.items():
        B, T, C, k, d = [int(v) for v in case["meta"]["BTCkd"]]
        sd = {"c.weight_v": torch.ones(2 * C, C, k), "c.weight_g": torch.full((2 * C, 1, 1), (C * k) ** 0.5),
              "c.bias": torch.zeros(2 * C)}
        x = torch.zeros(B, C, T) + torch.arange(0, T).float()
        y = O.conv1d(sd, "c", x, k, d, causal=True)
        close(y, case["out"]["0"], rtol=1e-6, atol=1e-5)


MODELS = G.load("models.npz")


@pytest.mark.parametrize("name", list(MODELS))
def test_full_model(name):
    case = MODELS[name]
    kw = G.kwargs_of(case)
    spec = spec_from_builder(kw.pop("builder"), **kw)
    sd = _leaf_sd(case)
    ins = G.tensors(case["in"])
    ins["mel"].requires_grad_(True)
    outs = O.model_forward(sd, spec, ins["text"], ins["mel"], ins.get("speaker_ids"),
                           ins["text_positions"], ins["frame_positions"],
                           case["meta"]["input_lengths"])
    _check_case(case, outs, sd, ins)


INCR = G.load("incremental.npz")


def _incremental_oracle(case, mode):
    """The oracle's stepwise decoder on one incremental fixture -> (outputs, alignments, dones (B,N,1), states)."""
    from oracle import dv3_incremental as OI
    kw = G.kwargs_of(case)
    bname = kw.pop("builder")
    fm = kw.pop("force_monotonic_attention")
    spec = spec_from_builder(bname, **kw)
    sd = G.tensors(case["sd"])
    ins = G.tensors(case["in"])
    common = dict(test_inputs=ins["mel"] if mode == "forced" else None, force_monotonic_attention=fm,
                  min_decoder_steps=int(case["meta"]["min_decoder_steps"]),
                  max_decoder_steps=int(case["meta"]["max_decoder_steps"]))
    enc = (ins["keys"], ins["values"])
    if bname == "nyanko":
        outs = OI.nyanko_decoder_incremental(sd, spec, enc, ins["text_positions"], **common)
    else:
        spk = None
        if "speaker_ids" in ins:
            spk = torch.nn.functional.embedding(ins["speaker_ids"], sd["embed_speakers.weight"])
        outs = OI.dv3_decoder_incremental(sd, spec, enc, ins["text_positions"], spk, **common)
    return outs[0], outs[1], torch.cat(outs[2], dim=1), outs[3]


@pytest.mark.parametrize("mode", ["forced", "free"])
@pytest.mark.parametrize("name", list(INCR))
def test_incremental_decoder(name, mode):
    """Inference path of the oracle (oracle/dv3_incremental.py) against the live reference's
    Decoder.incremental_forward, teacher-forced and free-running (same number of steps, same values)."""
    case = INCR[name]
    outs = _incremental_oracle(case, mode)
    for got, key in zip(outs, ("outputs", "alignments", "dones", "states")):
        assert tuple(got.shape) == tuple(case[mode][key].shape), key
        close(got, case[mode][key])


def test_audio_oracle_mel_basis_and_frames():
    """The one corroboration the reference tree offers for the (unpinned) audio path: its mel fixture of
    LJ001-0001 (212 893 samples) has 835 frames; and the Slaney filterbank equals torchaudio's."""
    from oracle import audio_oracle as A
    assert A.num_frames(212893) == 835
    assert A.num_frames(220500) == 865
    try:
        import torchaudio
    except Exception:
        pytest.skip("torchaudio not importable")
    ta = torchaudio.functional.melscale_fbanks(513, 125.0, 7600.0, 80, 22050, norm="slaney",
                                               mel_scale="slaney").T.numpy()
    np.testing.assert_allclose(A.mel_basis(), ta, rtol=1e-5, atol=1e-6)
    lin, mel = A.process_utterance(A.synthetic_clip(1, n=22050))
    assert lin.shape == (A.num_frames(22050), 513) and mel.shape == (A.num_frames(22050), 80)
    assert lin.min() >= 0 and lin.max() <= 1
