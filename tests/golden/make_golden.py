#!/usr/bin/env python
"""Generate the golden vectors in this directory from the LIVE reference implementation.

Runs only in the build container (needs /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference package is imported from a scratch copy under a temp dir (it needs a generated
``version.py``, reference setup.py:33-39 / deepvoice3_pytorch/__init__.py:3); nothing of it is
copied into this repository.  Every case stores: the module's state_dict (reference key names),
the seeded inputs, the reference outputs, and reference gradients of L = sum_i <out_i, R_i>
(R_i = cos(0.37*n + i), see loss_weights) w.r.t. inputs and parameters.  dropout = 0 throughout: the
reference's own parity tests run in .eval() (tests/test_deepvoice3.py:184-235) and bitwise Philox
parity with ATen is not a goal (SURVEY.md section 7).
"""
import os
import shutil
import sys
import tempfile
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
sys.path.insert(0, os.path.dirname(HERE))
import golden_util as G  # noqa: E402


def import_reference():
    tmp = tempfile.mkdtemp(prefix="dv3ref_")
    shutil.copytree(os.path.join(REF, "deepvoice3_pytorch"), os.path.join(tmp, "deepvoice3_pytorch"))
    with open(os.path.join(tmp, "deepvoice3_pytorch", "version.py"), "w") as f:
        f.write('__version__ = "0.1.1"\n')
    sys.path.insert(0, tmp)
    import deepvoice3_pytorch  # noqa: F401
    return tmp


def t2n(t):
    return t.detach().cpu().numpy()


class Fixture:
    def __init__(self):
        self.d = {}

    def put(self, case, group, name, value):
        self.d["%s|%s|%s" % (case, group, name)] = t2n(value) if torch.is_tensor(value) else np.asarray(value)

    def save(self, fname):
        G.save(fname, self.d)


def loss_weights(shape, i):
    """Deterministic, storage-free projection tensor R_i (tests rebuild it with the same formula)."""
    n = int(np.prod(shape))
    return torch.cos(torch.arange(n, dtype=torch.float64) * 0.37 + i).to(torch.float32).reshape(shape)


def run_case(fx, case, module, inputs, call, seed, meta=None):
    """inputs: dict name -> tensor (float tensors get requires_grad)."""
    for k, v in module.state_dict().items():
        fx.put(case, "sd", k, v)
    for k, v in (meta or {}).items():
        fx.put(case, "meta", k, v)
    leaves = {}
    for k, v in inputs.items():
        fx.put(case, "in", k, v)
        if torch.is_tensor(v) and v.is_floating_point():
            v = v.clone().requires_grad_(True)
        leaves[k] = v
    module.train()  # dropout=0 everywhere, so train == eval numerically but autograd is on
    outs = call(module, leaves)
    if torch.is_tensor(outs):
        outs = (outs,)
    loss = 0
    for i, o in enumerate(outs):
        fx.put(case, "out", str(i), o)
        loss = loss + (o * loss_weights(o.shape, i)).sum()
    module.zero_grad()
    loss.backward()
    for k, v in leaves.items():
        if torch.is_tensor(v) and v.requires_grad and v.grad is not None:
            fx.put(case, "gin", k, v.grad)
    for k, p in module.named_parameters():
        if p.grad is not None:
            fx.put(case, "gsd", k, p.grad)


def perturb(module, seed, scale=0.3):
    """Move g and bias away from their init (g=||v||, bias=0) so the fixtures exercise them."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in module.named_parameters():
            if n.endswith("weight_g"):
                p.mul_(1 + scale * torch.randn(p.shape, generator=g))
            elif n.endswith("bias"):
                p.add_(scale * torch.randn(p.shape, generator=g))


def block_cases():
    from deepvoice3_pytorch import modules as M
    from deepvoice3_pytorch.deepvoice3 import AttentionLayer
    fx = Fixture()
    gen = torch.Generator().manual_seed(1234)

    def rnd(*s):
        return torch.randn(*s, generator=gen)

    # --- BASELINE.json config #1: Conv1dGLU forward (B=2, C=64, T=128) and variants
    i = 0
    for (k, d, causal, residual) in [(3, 1, False, True), (3, 3, True, True), (3, 9, True, False),
                                     (3, 27, False, True), (5, 1, True, True), (5, 3, False, False),
                                     (1, 1, False, True), (2, 4, True, True)]:
        torch.manual_seed(100 + i)
        B, C, T = (2, 64, 128) if i < 2 else (2, 32, 72)   # i<2: BASELINE.json config #1 shape
        m = M.Conv1dGLU(1, None, C, C, k, dropout=0.0, dilation=d, causal=causal, residual=residual)
        perturb(m, 7 + i)
        run_case(fx, "glu%d" % i, m, {"x": rnd(B, C, T)}, lambda mod, L: mod(L["x"]), 50 + i,
                 meta=dict(k=k, d=d, causal=causal, residual=residual))
        i += 1
    # multi-speaker GLU: speaker embedding (B, T, 16) is genuinely time-varying in train mode
    for j, (k, d, causal, residual) in enumerate([(3, 1, True, True), (3, 3, False, True)]):
        torch.manual_seed(200 + j)
        m = M.Conv1dGLU(4, 16, 32, 32, k, dropout=0.0, dilation=d, causal=causal, residual=residual)
        perturb(m, 17 + j)
        run_case(fx, "glu_spk%d" % j, m, {"x": rnd(2, 32, 50), "spk": rnd(2, 50, 16)},
                 lambda mod, L: mod(L["x"], L["spk"]), 60 + j,
                 meta=dict(k=k, d=d, causal=causal, residual=residual))
    # ragged/odd sizes: T not a multiple of anything, C not a multiple of the tile
    for j, (Bc, Cc, Tc, k, d, causal) in enumerate([(3, 24, 37, 3, 9, True), (1, 40, 5, 3, 27, False),
                                                    (2, 8, 1, 3, 1, True)]):
        torch.manual_seed(300 + j)
        m = M.Conv1dGLU(1, None, Cc, Cc, k, dropout=0.0, dilation=d, causal=causal, residual=True)
        perturb(m, 27 + j)
        run_case(fx, "glu_odd%d" % j, m, {"x": rnd(Bc, Cc, Tc)}, lambda mod, L: mod(L["x"]), 70 + j,
                 meta=dict(k=k, d=d, causal=causal, residual=True))
    # --- HighwayConv1d
    for j, (k, d, causal) in enumerate([(3, 1, False), (3, 9, True), (1, 1, False), (3, 27, True)]):
        torch.manual_seed(400 + j)
        m = M.HighwayConv1d(32, 32, kernel_size=k, dilation=d, causal=causal, dropout=0.0)
        perturb(m, 37 + j)
        run_case(fx, "hw%d" % j, m, {"x": rnd(2, 32, 72)}, lambda mod, L: mod(L["x"]), 80 + j,
                 meta=dict(k=k, d=d, causal=causal))
    # --- weight-normed 1x1 Conv1d (odd widths 80 -> 48, and 513-like odd N), ConvTranspose1d, Linear
    for j, (cin, cout) in enumerate([(80, 48), (48, 65)]):
        torch.manual_seed(500 + j)
        m = M.Conv1d(cin, cout, 1, dropout=0.0)
        perturb(m, 47 + j)
        run_case(fx, "conv1x1_%d" % j, m, {"x": rnd(2, cin, 50)}, lambda mod, L: mod(L["x"]), 90 + j)
    torch.manual_seed(510)
    m = M.ConvTranspose1d(32, 48, 2, padding=0, stride=2)
    perturb(m, 57)
    run_case(fx, "convT", m, {"x": rnd(2, 32, 25)}, lambda mod, L: mod(L["x"]), 95)
    torch.manual_seed(520)
    m = M.Linear(16, 64)
    perturb(m, 58)
    run_case(fx, "linear", m, {"x": rnd(2, 30, 16)}, lambda mod, L: mod(L["x"]), 96)
    # --- AttentionLayer with / without projections and mask
    for j, (kp, vp, masked) in enumerate([(True, True, True), (False, False, False), (True, False, True)]):
        torch.manual_seed(600 + j)
        m = AttentionLayer(48, 32, dropout=0.0, key_projection=kp, value_projection=vp)
        perturb(m, 67 + j)
        Bq, Td, Ts = 3, 20, 13
        lengths = np.array([13, 7, 10])
        mask = ~(torch.arange(Ts)[None, :] < torch.tensor(lengths)[:, None]) if masked else None
        ins = {"query": rnd(Bq, Td, 48), "keys": 0.3 * rnd(Bq, 32, Ts), "values": rnd(Bq, Ts, 32)}
        run_case(fx, "attn%d" % j, m, ins,
                 lambda mod, L, mask=mask: mod(L["query"], (L["keys"], L["values"]), mask=mask),
                 100 + j, meta=dict(lengths=lengths if masked else np.zeros(0)))
    # --- SinusoidalEncoding (reference tests/test_embedding.py) incl. per-utterance rates
    for j, w in enumerate([1.0, 0.5, 2.0, 10.0, 20.0, 1.29, 7.6]):
        m = M.SinusoidalEncoding(160, 64)
        x = torch.arange(0, 128).long()[None, :].repeat(2, 1)
        x[1, 100:] = 0
        fx.put("sin%d" % j, "meta", "w", w)
        fx.put("sin%d" % j, "in", "x", x)
        fx.put("sin%d" % j, "out", "0", m(x, w))
        fx.put("sin%d" % j, "out", "table", M.position_encoding_init(160, 64, position_rate=w))
    m = M.SinusoidalEncoding(64, 32)
    x = torch.tensor([[1, 2, 3, 4, 0, 0], [1, 2, 3, 4, 5, 6], [5, 9, 63, 0, 1, 1]])
    wv = torch.tensor([0.7, 1.9, 3.3])
    fx.put("sin_batch", "in", "x", x)
    fx.put("sin_batch", "meta", "w", wv)
    fx.put("sin_batch", "out", "0", m(x, wv))
    fx.put("sin_batch", "sd", "weight", m.weight)
    fx.save("blocks.npz")


def model_cases():
    from deepvoice3_pytorch import builder
    common = dict(n_vocab=149, mel_dim=80, padding_idx=0, dropout=0.0, max_positions=64)
    cases = {
        # reference tests/test_deepvoice3.py:27-46 topology (k=5, downsample_step=1) but r=1: with r=4 the
        # reference's own mel_outputs.view(B,-1,mel_dim) (__init__.py:83) raises on torch 2.11
        # (sigmoid of a transposed tensor is no longer viewable) -- reference rot, not our path.
        "dv3_k5": ("deepvoice3", dict(embed_dim=16, linear_dim=33, r=1, kernel_size=5,
                                      encoder_channels=8, decoder_channels=16, converter_channels=16,
                                      use_memory_mask=True, key_projection=True, value_projection=True)),
        # ljspeech-preset topology (k=3, r=1, ds=4 => two ConvTranspose upsamplers), narrow
        "dv3_lj": ("deepvoice3", dict(embed_dim=16, linear_dim=33, r=1, downsample_step=4,
                                      kernel_size=3, encoder_channels=24, decoder_channels=16,
                                      converter_channels=16, use_memory_mask=True,
                                      key_projection=True, value_projection=True)),
        # vctk-preset topology
        "dv3_ms": ("deepvoice3_multispeaker", dict(embed_dim=16, linear_dim=33, r=1, downsample_step=4,
                                                   kernel_size=3, encoder_channels=24,
                                                   decoder_channels=16, converter_channels=16,
                                                   n_speakers=5, speaker_embed_dim=16,
                                                   use_memory_mask=True)),
        "nyanko": ("nyanko", dict(embed_dim=12, linear_dim=33, r=1, downsample_step=4, kernel_size=3,
                                  encoder_channels=16, decoder_channels=16, converter_channels=20,
                                  use_memory_mask=True)),
    }
    fx = Fixture()
    for ci, (name, (bname, kw)) in enumerate(cases.items()):
        torch.manual_seed(1000 + ci)
        kw = dict(common, **kw)
        model = getattr(builder, bname)(**kw)
        perturb(model, 77 + ci, scale=0.2)
        gen = torch.Generator().manual_seed(2000 + ci)
        B, Ttext = 3, 11
        r, ds = kw["r"], kw.get("downsample_step", 1)
        Tdec = 8
        lengths = np.array([11, 6, 9])
        text = torch.randint(2, 149, (B, Ttext), generator=gen)
        text_pos = torch.arange(1, Ttext + 1)[None, :].repeat(B, 1)
        for b in range(B):
            text[b, lengths[b]:] = 0
            text_pos[b, lengths[b]:] = 0
        mel = torch.rand(B, Tdec * r, 80, generator=gen)
        frame_pos = torch.arange(1, Tdec + 1)[None, :].repeat(B, 1)
        ins = {"text": text, "mel": mel, "text_positions": text_pos, "frame_positions": frame_pos}
        spk = None
        if kw.get("n_speakers", 1) > 1:
            spk = torch.tensor([0, 3, 4])
            ins["speaker_ids"] = spk
        for k_, v_ in kw.items():
            fx.put(name, "kw", k_, v_)
        fx.put(name, "kw", "builder", bname)
        run_case(fx, name, model, ins,
                 lambda mod, L, spk=spk, lengths=lengths: mod(
                     L["text"], L["mel"], speaker_ids=spk, text_positions=L["text_positions"],
                     frame_positions=L["frame_positions"], input_lengths=lengths),
                 3000 + ci, meta=dict(input_lengths=lengths))
    fx.save("models.npz")


def incremental_cases():
    """Inference path: Decoder.incremental_forward (reference deepvoice3.py:367-485, nyanko.py:250-338) teacher-forced
    (``test_inputs``) and free-running, through the reference's own call stack in .eval().  Decoders get a small
    max_decoder_steps so the free run stops on the step cap or on the done flags.  Stored: the state_dict, the
    text / positions / speaker ids, the encoder output the decoder consumed, and the four returned values
    (outputs, alignments, dones stacked, decoder_states) of both modes; plus the whole-model inference call."""
    from deepvoice3_pytorch import builder
    common = dict(n_vocab=149, mel_dim=80, padding_idx=0, dropout=0.0, max_positions=64)
    cases = {
        "inc_dv3": ("deepvoice3", dict(embed_dim=16, linear_dim=33, r=1, downsample_step=4, kernel_size=3,
                                       encoder_channels=24, decoder_channels=16, converter_channels=16,
                                       key_projection=True, value_projection=True,
                                       force_monotonic_attention=True), 2),
        "inc_dv3_k5_free": ("deepvoice3", dict(embed_dim=16, linear_dim=33, r=1, kernel_size=5,
                                               encoder_channels=8, decoder_channels=16, converter_channels=16,
                                               key_projection=False, value_projection=False,
                                               force_monotonic_attention=False), 2),
        # the reference's incremental speaker path broadcasts (B,1,C) + (B,C): only B = 1 is meaningful
        "inc_dv3_ms": ("deepvoice3_multispeaker", dict(embed_dim=16, linear_dim=33, r=1, downsample_step=4,
                                                       kernel_size=3, encoder_channels=24, decoder_channels=16,
                                                       converter_channels=16, n_speakers=5, speaker_embed_dim=16,
                                                       force_monotonic_attention=True), 1),
        "inc_nyanko": ("nyanko", dict(embed_dim=12, linear_dim=33, r=1, downsample_step=4, kernel_size=3,
                                      encoder_channels=16, decoder_channels=16, converter_channels=20,
                                      force_monotonic_attention=True), 2),
    }
    fx = Fixture()
    for ci, (name, (bname, kw, B)) in enumerate(cases.items()):
        torch.manual_seed(5000 + ci)
        kw = dict(common, **kw)
        model = getattr(builder, bname)(**kw)
        perturb(model, 177 + ci, scale=0.2)
        model.eval()
        dec = model.seq2seq.decoder
        dec.max_decoder_steps, dec.min_decoder_steps = 14, 3
        gen = torch.Generator().manual_seed(6000 + ci)
        Ttext, Tdec = 9, 12
        text = torch.randint(2, 149, (B, Ttext), generator=gen)
        text_pos = torch.arange(1, Ttext + 1)[None, :].repeat(B, 1)
        mel = torch.rand(B, Tdec, 80, generator=gen)
        spk_ids = torch.tensor([3]) if kw.get("n_speakers", 1) > 1 else None
        for k_, v_ in kw.items():
            fx.put(name, "kw", k_, v_)
        fx.put(name, "kw", "builder", bname)
        for k_, v_ in model.state_dict().items():
            fx.put(name, "sd", k_, v_)
        fx.put(name, "in", "text", text)
        fx.put(name, "in", "text_positions", text_pos)
        fx.put(name, "in", "mel", mel)
        if spk_ids is not None:
            fx.put(name, "in", "speaker_ids", spk_ids)
        fx.put(name, "meta", "max_decoder_steps", dec.max_decoder_steps)
        fx.put(name, "meta", "min_decoder_steps", dec.min_decoder_steps)
        with torch.no_grad():
            spk = model.embed_speakers(spk_ids) if spk_ids is not None else None
            if bname == "nyanko":
                enc = model.seq2seq.encoder(text)
            else:
                enc = model.seq2seq.encoder(text, speaker_embed=spk)
            fx.put(name, "in", "keys", enc[0])
            fx.put(name, "in", "values", enc[1])
            for mode in ("forced", "free"):
                dec.start_fresh_sequence()
                args = (enc, text_pos) if bname == "nyanko" else (enc, text_pos, spk)
                outs = dec.incremental_forward(*args, test_inputs=mel if mode == "forced" else None)
                outputs, alignments, dones, states = outs
                fx.put(name, mode, "outputs", outputs)
                fx.put(name, mode, "alignments", alignments)
                fx.put(name, mode, "dones", torch.cat(dones, dim=1))      # (B, N, 1)
                fx.put(name, mode, "states", states)
            # the user-facing inference call (reference synthesis.py:62-64)
            mel_o, lin_o, ali_o, done_o = model(text, text_positions=text_pos, speaker_ids=spk_ids)
            fx.put(name, "model", "mel", mel_o)
            fx.put(name, "model", "linear", lin_o)
            fx.put(name, "model", "alignments", ali_o)
            fx.put(name, "model", "dones", torch.cat(done_o, dim=1))
        print(name, "forced", tuple(fx.d[name + "|forced|outputs"].shape), "free",
              tuple(fx.d[name + "|free|outputs"].shape))
    fx.save("incremental.npz")


def conv_ramp_case():
    """reference tests/test_conv.py:10-63: causal conv, weights 1, bias 0, ramp input -> exact ints."""
    fx = Fixture()
    from torch import nn
    i = 0
    for B in [1, 4]:
        for T in [5, 10]:
            for C in [1, 2, 4]:
                for k in [2, 3]:
                    for d in [1, 2, 3, 4, 5, 9, 27]:
                        conv = nn.Conv1d(C, 2 * C, k, padding=(k - 1) * d, dilation=d)
                        conv.weight.data.fill_(1.0)
                        conv.bias.data.zero_()
                        x = torch.zeros(B, C, T) + torch.arange(0, T).float()
                        y = conv(x)[:, :, :T]
                        fx.put("ramp%d" % i, "meta", "BTCkd", np.array([B, T, C, k, d]))
                        fx.put("ramp%d" % i, "out", "0", y)
                        i += 1
    fx.save("conv_ramp.npz")


def init_fingerprints():
    """Same torch seed -> same initial weights: per-tensor (sum, abs-sum, first element) of the reference
    builders' freshly initialised models at the three BASELINE.json presets (seed 4321)."""
    from deepvoice3_pytorch import builder
    from test_gpu_models import preset_kwargs
    fx = Fixture()
    for preset in ["deepvoice3_ljspeech", "nyanko_ljspeech", "deepvoice3_vctk"]:
        bname, kw = preset_kwargs(preset)
        torch.manual_seed(4321)
        sd = getattr(builder, bname)(dropout=0.05, **kw).state_dict()
        fx.put(preset, "meta", "keys", np.array(list(sd.keys())))
        fx.put(preset, "meta", "shapes", np.array([str(tuple(v.shape)) for v in sd.values()]))
        fx.put(preset, "out", "fingerprint", np.array(
            [[float(v.double().sum()), float(v.double().abs().sum()), float(v.flatten()[0])]
             for v in sd.values()]))
    fx.save("init_fingerprints.npz")


if __name__ == "__main__":
    tmp = import_reference()
    try:
        torch.set_num_threads(1)  # deterministic reduction order
        only = set(sys.argv[1:])      # e.g. `make_golden.py incremental` regenerates that one fixture
        for name, fn in (("blocks", block_cases), ("models", model_cases), ("conv_ramp", conv_ramp_case),
                         ("init_fingerprints", init_fingerprints), ("incremental", incremental_cases)):
            if not only or name in only:
                fn()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
