"""CPU-only checks of the host side: the C-ABI library exports what include/dv3b200.h declares, the builder
API mirrors the reference (keys, shapes, seed-for-seed initialisation, error behaviour), and the product path
refuses to run without CUDA (no CPU fallback)."""
import ctypes

import numpy as np
import pytest
import torch

import golden_util as G
from test_gpu_models import preset_kwargs


@pytest.fixture(scope="session", autouse=True)
def built_library():
    from deepvoice3_pytorch_b200 import _build
    _build.build()


def test_library_exports_every_declared_symbol():
    from deepvoice3_pytorch_b200._lib import parse_header, LIB_PATH
    decls = parse_header()
    assert len(decls) >= 20
    dll = ctypes.CDLL(LIB_PATH)
    for name in decls:
        assert hasattr(dll, name), "libdv3b200.so lacks %s declared in include/dv3b200.h" % name
    assert dll.dv3_abi_version() >= 1


@pytest.mark.parametrize("preset", ["deepvoice3_ljspeech", "nyanko_ljspeech", "deepvoice3_vctk"])
def test_state_dict_and_init_match_reference(preset):
    """Same keys in the same order, same shapes and -- for the same torch seed -- the same initial values as the
    reference builder (fingerprints recorded from the live reference by tests/golden/make_golden.py)."""
    from deepvoice3_pytorch_b200 import builder
    fp = G.load("init_fingerprints.npz")[preset]
    bname, kw = preset_kwargs(preset)
    torch.manual_seed(4321)
    sd = getattr(builder, bname)(dropout=0.05, **kw).state_dict()
    assert list(sd.keys()) == [str(k) for k in fp["meta"]["keys"]]
    assert [str(tuple(v.shape)) for v in sd.values()] == [str(s) for s in fp["meta"]["shapes"]]
    got = np.array([[float(v.double().sum()), float(v.double().abs().sum()), float(v.flatten()[0])]
                    for v in sd.values()])
    np.testing.assert_allclose(got, fp["out"]["fingerprint"], rtol=1e-12, atol=0)


def test_builder_error_behaviour():
    from deepvoice3_pytorch_b200 import builder
    with pytest.raises(ValueError):
        builder.nyanko(n_vocab=149, n_speakers=2)                       # reference builder.py:120-121
    with pytest.raises(ValueError):
        builder.nyanko(n_vocab=149, downsample_step=1, r=1)             # reference builder.py:122-123
    with pytest.raises(AssertionError):
        builder.nyanko(n_vocab=149, encoder_channels=64, decoder_channels=32)


def test_trainable_parameters_exclude_position_tables():
    from deepvoice3_pytorch_b200 import builder
    m = builder.deepvoice3(n_vocab=149, embed_dim=16, r=1, downsample_step=4, kernel_size=3,
                           encoder_channels=16, decoder_channels=16, converter_channels=16, linear_dim=33)
    ids = set(map(id, m.get_trainable_parameters()))
    dec = m.seq2seq.decoder
    assert id(dec.embed_query_positions.weight) not in ids and id(dec.embed_keys_positions.weight) not in ids
    assert id(m.seq2seq.encoder.embed_tokens.weight) in ids
    m.trainable_positional_encodings = True
    assert id(dec.embed_query_positions.weight) in set(map(id, m.get_trainable_parameters()))


def test_memory_mask_is_bit_exact():
    from deepvoice3_pytorch_b200.modules import get_mask_from_lengths
    lengths = np.array([5, 1, 3])
    mask = get_mask_from_lengths(torch.zeros(3, 5, 2), lengths)
    want = np.array([[0, 0, 0, 0, 0], [0, 1, 1, 1, 1], [0, 0, 0, 1, 1]], dtype=bool)
    assert mask.dtype == torch.bool and np.array_equal(mask.numpy(), want)


def test_position_table_is_bit_exact():
    from deepvoice3_pytorch_b200.modules import position_encoding_init, SinusoidalEncoding
    blocks = G.load("blocks.npz")
    for j in range(7):
        case = blocks["sin%d" % j]
        w = float(case["meta"]["w"])
        n, d = case["out"]["table"].shape
        assert np.array_equal(position_encoding_init(n, d, position_rate=w).numpy(), case["out"]["table"])
    assert np.array_equal(SinusoidalEncoding(64, 32).weight.detach().numpy(), blocks["sin_batch"]["sd"]["weight"])


def test_no_cpu_fallback():
    """The product path must fail loudly without CUDA tensors -- never route through a CPU implementation."""
    from deepvoice3_pytorch_b200 import ops
    from deepvoice3_pytorch_b200._lib import Dv3Error
    x = torch.zeros(1, 4, 8)
    v = torch.ones(8, 4, 3)
    g = torch.ones(8, 1, 1)
    with pytest.raises(Dv3Error):
        ops.convblock(x, v, g, torch.zeros(8))
    with pytest.raises(Dv3Error):
        ops.transpose12(x)


def test_product_never_imports_oracle():
    import os
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "deepvoice3_pytorch_b200")
    for dirpath, _, files in os.walk(root):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_abi_structs_match_the_c_header(tmp_path):
    """The structs that cross the C ABI by pointer (Dv3WnEntry, Dv3IncStep, Dv3IncAttn) are mirrored by hand in
    ctypes; compile the header with gcc and compare sizeof / every field offset."""
    import ctypes
    import os
    import subprocess
    from deepvoice3_pytorch_b200.weight_bank import Dv3WnEntry
    from deepvoice3_pytorch_b200.incremental import Dv3IncStep, Dv3IncAttn
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {"Dv3WnEntry": Dv3WnEntry, "Dv3IncStep": Dv3IncStep, "Dv3IncAttn": Dv3IncAttn}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dv3b200.h"', 'int main(void) {']
    for name, st in structs.items():
        lines.append('printf("%s sizeof %%zu\\n", sizeof(%s));' % (name, name))
        for fname, _ in st._fields_:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (name, fname, name, fname))
    lines += ['return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    for line in out.strip().splitlines():
        name, field, value = line.split()
        st = structs[name]
        got = ctypes.sizeof(st) if field == "sizeof" else getattr(st, field).offset
        assert got == int(value), "%s.%s: ctypes %d vs C %s" % (name, field, got, value)


def test_tc_gemm_entry_points_refuse_a_non_null_reserved_argument():
    """dv3_tc_convblock_fwd and dv3_tc_conv keep a `reserved` pointer slot in front of `stream`, which must be NULL.
    Any other value is refused before any device work, so a caller that passes a stream or a pointer there gets an
    error rather than a launch on the wrong stream."""
    from deepvoice3_pytorch_b200._lib import lib
    bad = ctypes.c_void_p(16)
    rc = lib.raw("dv3_tc_convblock_fwd")(None, None, 2, None, None, None, None, None, None, 1, 128, 128, 3, 1, 0, 0, 1,
                                         bad, None)
    assert rc != 0 and "must be NULL" in lib.raw("dv3_last_error")().decode()
    rc = lib.raw("dv3_tc_conv")(None, None, 2, None, 1, 128, 128, 128, 1, 1, 0, 0, None, 0, 0.0, None, 0, 0, None, None,
                                0.0, bad, None)
    assert rc != 0 and "must be NULL" in lib.raw("dv3_last_error")().decode()


def test_incremental_stop_rule_matches_reference_loop():
    """Host logic of the free-running decoder: the number of steps derived from the done flags equals what the
    reference's while-loop does (break after step n if all(done > .5) and n > min_steps, or n > max_steps;
    deepvoice3.py:466-470)."""
    import torch
    from deepvoice3_pytorch_b200.incremental import _stop_step

    def reference(done, min_steps, max_steps):
        t = 0
        while t < done.size(1):
            d = done[:, t]
            t += 1
            if bool((d > 0.5).all()) and t > min_steps:
                return t
            elif t > max_steps:
                return t
        return None

    gen = torch.Generator().manual_seed(0)
    for _ in range(200):
        n = int(torch.randint(1, 40, (1,), generator=gen))
        done = torch.rand(3, n, generator=gen) ** 0.2
        mn, mx = int(torch.randint(0, 12, (1,), generator=gen)), int(torch.randint(5, 45, (1,), generator=gen))
        assert _stop_step(done, mn, mx) == reference(done, mn, mx)


def test_hparams_mapping_matches_the_bench_presets():
    """hparams.builder_kwargs restates reference train.py:812-840; applied to the values of the reference's
    presets/*.json (copied below: they are data) it must give exactly the builder kwargs bench.py hard-codes for the
    BASELINE.json presets, and train_step_kwargs must give the optimiser / loss settings of train.py."""
    import bench
    from deepvoice3_pytorch_b200 import hparams
    from deepvoice3_pytorch_b200.train_step import noam_learning_rate_decay
    common = dict(adam_beta1=0.5, adam_beta2=0.9, adam_eps=1e-6, binary_divergence_weight=0.1, clip_thresh=0.1,
                  converter_channels=256, decoder_channels=256, downsample_step=4, dropout=0.050000000000000044,
                  fft_size=1024, force_monotonic_attention=True, freeze_embedding=False, initial_learning_rate=0.0005,
                  kernel_size=3, lr_schedule="noam_learning_rate_decay", lr_schedule_kwargs={}, masked_loss_weight=0.5,
                  num_mels=80, outputs_per_step=1, padding_idx=0, speaker_embed_dim=16,
                  trainable_positional_encodings=False, use_decoder_state_for_postnet_input=True,
                  use_guided_attention=True, use_memory_mask=True, window_ahead=3, window_backward=1,
                  key_position_rate=1.385, query_position_rate=1.0, embedding_weight_std=0.1)
    presets = {
        "deepvoice3_ljspeech": dict(common, builder="deepvoice3", encoder_channels=512, text_embed_dim=256, n_speakers=1,
                                    max_positions=512, speaker_embedding_weight_std=0.01, key_projection=True,
                                    value_projection=True, guided_attention_sigma=0.2),
        "nyanko_ljspeech": dict(common, builder="nyanko", encoder_channels=256, text_embed_dim=128, n_speakers=1,
                                max_positions=512, speaker_embedding_weight_std=0.01, key_projection=False,
                                value_projection=False, guided_attention_sigma=0.2),
        "deepvoice3_vctk": dict(common, builder="deepvoice3_multispeaker", encoder_channels=512, text_embed_dim=256,
                                n_speakers=108, max_positions=1024, speaker_embedding_weight_std=0.05,
                                key_projection=True, value_projection=True, guided_attention_sigma=0.4,
                                key_position_rate=7.6, query_position_rate=2.0),
    }
    for name, hp in presets.items():
        bname, kw = hparams.builder_kwargs(hp, n_vocab=149)
        want_name, want_kw, extra = bench.PRESETS[name]
        assert bname == want_name
        assert set(kw) == set(want_kw)
        for k in kw:
            assert kw[k] == pytest.approx(want_kw[k]), (name, k)
        ts = hparams.train_step_kwargs(hp)
        assert ts["guided_attention_sigma"] == extra["guided_attention_sigma"]
        assert ts["betas"] == (0.5, 0.9) and ts["eps"] == 1e-6 and ts["clip_thresh"] == 0.1
        assert ts["lr_schedule"] is noam_learning_rate_decay and ts["init_lr"] == 5e-4
    model = hparams.build_model(dict(presets["nyanko_ljspeech"], encoder_channels=32, decoder_channels=32,
                                     converter_channels=32, text_embed_dim=16), n_vocab=149)
    assert model.seq2seq.decoder.in_dim == 80 and model.linear_dim == 513


def test_audio_file_helpers_round_trip(tmp_path):
    """audio.load_wav / save_wav / preemphasis / _linear_to_mel: the host-side helpers of reference audio.py:12-23,64-68
    (scipy only).  save -> load reproduces the peak-normalised 16-bit signal; a file at another rate is resampled to
    hparams.sample_rate; preemphasis matches the oracle's restatement."""
    from deepvoice3_pytorch_b200 import audio
    from oracle import audio_oracle as A
    from scipy.io import wavfile
    rng = np.random.RandomState(0)
    x = (0.3 * rng.randn(4000)).astype(np.float32)
    p = str(tmp_path / "a.wav")
    audio.save_wav(x, p)
    sr, raw = wavfile.read(p)
    assert sr == audio.hparams.sample_rate and raw.dtype == np.int16 and abs(int(np.abs(raw).max()) - 32767) <= 1
    y = audio.load_wav(p)
    assert y.dtype == np.float32 and y.shape == x.shape
    np.testing.assert_allclose(y, x / np.abs(x).max() * (32767 / 32768.0), atol=1.0 / 32768)
    wavfile.write(str(tmp_path / "b.wav"), 44100, np.stack([raw, raw], axis=1).repeat(2, axis=0)[:8000])   # stereo, 2x rate
    z = audio.load_wav(str(tmp_path / "b.wav"))
    assert z.ndim == 1 and abs(len(z) - 4000) <= 1
    np.testing.assert_allclose(audio.preemphasis(x), A.preemphasis(x.astype(np.float64)), atol=1e-6)
    S = np.abs(rng.randn(513, 7)).astype(np.float32)
    np.testing.assert_allclose(audio._linear_to_mel(S), A.mel_basis() @ S, rtol=1e-5, atol=1e-7)
