"""The drop-in claim, exercised against what the reference's OWN ``train.py``, ``synthesis.py`` and ``ljspeech.py``
produced on the reference package (tests/golden/dropin.*.npz, written by tests/golden/make_dropin_golden.py): this
package, driven the way those callers drive a model -- ``build_model()`` from the reference's hyper-parameters,
``collate_fn`` batches, ``model(...)``, the train loop's losses, ``loss.backward()``, ``clip_grad_norm_`` and
``torch.optim.Adam``; ``tts()``; ``_process_utterance`` -- gives the same weights, losses and outputs."""
import hashlib
import json

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import golden_util as G
from oracle import ref_harness as H

DROPIN = G.load("dropin.npz")


def _hparams(preset):
    """The reference's hparams after presets/<preset>.json (train.py:936-939)."""
    return json.loads(str(DROPIN[preset]["meta"]["hparams"]))


def _build_model(hp):
    """train.py:812-840 ``build_model()`` on this package, seed 0."""
    from deepvoice3_pytorch_b200 import hparams
    torch.manual_seed(0)
    return hparams.build_model(hp, n_vocab=H.N_VOCAB)


def test_train_py_build_model_on_this_package_cpu():
    """``build_model()`` from the reference's deepvoice3_ljspeech hyper-parameters: same class surface, same state_dict
    keys and shapes and -- for the same seed -- bit-identical initial weights as on the reference package."""
    model = _build_model(_hparams("deepvoice3_ljspeech"))
    assert hasattr(model, "get_trainable_parameters") and hasattr(model.seq2seq.decoder, "max_decoder_steps")
    assert type(model).__module__.startswith("deepvoice3_pytorch_b200")
    case = DROPIN["build_model"]
    sd = model.state_dict()
    assert list(sd.keys()) == [str(k) for k in case["meta"]["keys"]]
    assert [str(tuple(v.shape)) for v in sd.values()] == [str(s) for s in case["meta"]["shapes"]]
    for (k, v), want in zip(sd.items(), case["out"]["sha256"]):
        assert hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() == str(want), k


@pytest.mark.gpu
@pytest.mark.parametrize("preset,n_speakers", [("deepvoice3_ljspeech", 1), ("nyanko_ljspeech", 1),
                                               ("deepvoice3_vctk", 108)])
def test_reference_train_loop_runs_unchanged_on_this_package(preset, n_speakers):
    """4 optimizer steps of the reference ``train()`` loop (train.py:604-785: noam learning rate, model(...), the
    mel / done / linear / guided-attention losses, clip_grad_norm_, torch.optim.Adam) on synthetic utterances batched
    like ``collate_fn``, on this package (default tensor-core mode, eager), against the scalars the reference package
    logged for the same loop and data.  dropout = 0 so the two are comparable."""
    from deepvoice3_pytorch_b200 import hparams
    from deepvoice3_pytorch_b200 import train_step as TS
    from deepvoice3_pytorch_b200.data import collate
    hp = _hparams(preset)
    hp["dropout"] = 0.0
    kw = hparams.train_step_kwargs(hp)
    r, ds, mw, w = kw["r"], kw["downsample_step"], kw["masked_loss_weight"], kw["binary_divergence_weight"]
    model = _build_model(hp).to("cuda")
    opt = torch.optim.Adam(model.get_trainable_parameters(), lr=kw["init_lr"], betas=kw["betas"], eps=kw["eps"])
    utts = H.synthetic_utterances(16, seed=3, n_speakers=n_speakers, min_text=40, max_text=100, min_frames=200,
                                  max_frames=400)
    logs = {tag: [] for tag in ("loss", "mel_l1_loss", "linear_l1_loss", "done_loss", "attn_loss", "gradient_norm")}
    for step in range(4):
        host = collate(utts[4 * step:4 * step + 4], r=r, downsample_step=ds)
        b = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in host.items()}
        for group in opt.param_groups:
            group["lr"] = kw["lr_schedule"](kw["init_lr"], step)
        model.train()
        opt.zero_grad()
        mel_out, lin_out, attn, done_hat = model(b["x"], b["mel"], speaker_ids=b.get("speaker_ids"),
                                                 text_positions=b["text_positions"],
                                                 frame_positions=b["frame_positions"], input_lengths=b["input_lengths"])
        mel, y, tl = b["mel"], b["y"], b["target_lengths"]
        dec_mask = tgt_mask = None
        if mw > 0:
            dec_mask = TS.sequence_mask(tl // (r * ds), mel.size(1)).unsqueeze(-1)
            tgt_mask = TS.sequence_mask(tl, y.size(1)).unsqueeze(-1) if ds > 1 else dec_mask
            dec_mask, tgt_mask = dec_mask[:, r:, :], tgt_mask[:, r:, :]
        mel_l1, mel_bd = TS.spec_loss(mel_out[:, :-r, :], mel[:, r:, :], dec_mask, mw, w)
        done_loss = F.binary_cross_entropy(done_hat, b["done"])
        lin_l1, lin_bd = TS.spec_loss(lin_out[:, :-r, :], y[:, r:, :], tgt_mask, mw, w,
                                      priority_bin=TS.priority_bin_of(kw["priority_freq"], kw["sample_rate"],
                                                                      lin_out.size(-1)),
                                      priority_w=kw["priority_freq_weight"])
        soft = TS.guided_attention_mask(b["input_lengths_dev"], tl // r // ds, attn.size(-2), attn.size(-1),
                                        kw["guided_attention_sigma"])
        attn_loss = (attn * soft).mean()
        loss = (1 - w) * mel_l1 + w * mel_bd + done_loss + (1 - w) * lin_l1 + w * lin_bd + attn_loss
        loss.backward()
        grad_norm = torch.nn.utils.clip_grad_norm_(model.get_trainable_parameters(), kw["clip_thresh"])
        opt.step()
        for tag, v in (("loss", loss), ("mel_l1_loss", mel_l1), ("linear_l1_loss", lin_l1), ("done_loss", done_loss),
                       ("attn_loss", attn_loss), ("gradient_norm", grad_norm)):
            logs[tag].append(float(v.detach()))
    ref = DROPIN["train_" + preset]["out"]
    for tag, got in logs.items():
        got, want = np.array(got), ref[tag]
        assert len(want) == 4 and len(got) == 4, tag
        np.testing.assert_allclose(got[0], want[0], rtol=2e-4, err_msg=tag + " (first step: identical weights)")
        np.testing.assert_allclose(got, want, rtol=5e-3, err_msg=tag)
    assert all(np.isfinite(logs["loss"]))


@pytest.mark.gpu
def test_reference_synthesis_tts_runs_unchanged_on_this_package():
    """The inference-side caller: reference ``synthesis.py:tts()`` (text ids -> ``model(...)`` autoregressive decoding
    -> ``audio._denormalize`` / ``audio.inv_spectrogram``) with this package's model and ``audio`` module, against
    what the same function returned on the reference package.  Same weights, a decoder that never raises the done flag
    early, 24 decoder steps: mel / linear / alignment agree; the waveform is finite and of the length the frame count
    implies, the length the reference produced."""
    from deepvoice3_pytorch_b200 import audio
    model = _build_model(_hparams("deepvoice3_ljspeech"))
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    sd["seq2seq.decoder.fc.bias"] = torch.full_like(sd["seq2seq.decoder.fc.bias"], -8.0)   # never "done"
    model.load_state_dict(sd)
    model.seq2seq.decoder.max_decoder_steps = 24
    old_iters = audio.hparams.griffin_lim_iters
    audio.hparams.griffin_lim_iters = 4
    try:
        model = model.to("cuda")
        model.eval()
        model.make_generation_fast_()
        sequence = torch.from_numpy(np.array(H.CharFrontend.text_to_sequence("hello b200", p=0)))
        sequence = sequence.unsqueeze(0).long().cuda()
        text_positions = torch.arange(1, sequence.size(-1) + 1).unsqueeze(0).long().cuda()
        with torch.no_grad():
            mel_outputs, linear_outputs, alignments, done = model(sequence, text_positions=text_positions,
                                                                  speaker_ids=None)
        linear_output = linear_outputs[0].cpu().numpy()
        got = {"spectrogram": audio._denormalize(linear_output), "alignment": alignments[0].cpu().numpy(),
               "mel": audio._denormalize(mel_outputs[0].cpu().numpy())}
        waveform = np.asarray(audio.inv_spectrogram(linear_output.T))
    finally:
        audio.hparams.griffin_lim_iters = old_iters
    assert type(model).__module__.startswith("deepvoice3_pytorch_b200")
    ref = DROPIN["tts"]
    for name in ("alignment", "spectrogram", "mel"):
        r, g = ref["out"][name], got[name]
        assert r.shape == g.shape, name
        scale = max(1.0, float(np.abs(r).max()))
        np.testing.assert_allclose(g, r, rtol=2e-3, atol=2e-3 * scale, err_msg=name)
    T = ref["out"]["spectrogram"].shape[0]
    assert got["spectrogram"].shape == (T, 513) and got["mel"].shape[1] == 80
    n = audio.inv_num_samples(T)
    assert waveform.shape == (n,) and np.isfinite(waveform).all() and np.abs(waveform).max() > 0
    assert int(ref["meta"]["waveform_len"]) == n


@pytest.mark.gpu
def test_reference_ljspeech_preprocessor_and_batched_equivalent(tmp_path):
    """The caller of the audio front-end: reference ``ljspeech.py:_process_utterance`` (load_wav -> spectrogram ->
    melspectrogram -> np.save, :40-79) on this package's ``audio`` module, one clip per launch, writes the same files
    as the batched ``preprocess.build_from_path`` (same arguments, one fused launch per batch), bit for bit; and
    ``build_from_path`` returns the ``train.txt`` rows the reference returned, including its skip of short
    transcripts."""
    from scipy.io import wavfile
    from oracle import audio_oracle as A
    from deepvoice3_pytorch_b200 import audio, preprocess
    hp = _hparams("deepvoice3_ljspeech")
    assert hp["min_text"] == audio.hparams.min_text and not hp["rescaling"]
    in_dir, out_b = tmp_path / "in", tmp_path / "ours"
    (in_dir / "wavs").mkdir(parents=True)
    out_b.mkdir()
    lens = [30001, 22050, 5000, 47777, 12345]
    texts = ["the quick brown fox jumps over the lazy dog %d" % i for i in range(5)]
    texts[2] = "too short"                                  # < hparams.min_text = 20: skipped by both
    with open(in_dir / "metadata.csv", "w", encoding="utf-8") as f:
        for i, (n, t) in enumerate(zip(lens, texts)):
            x = A.synthetic_clip(70 + i, n=n)
            wavfile.write(str(in_dir / "wavs" / ("LJ%03d.wav" % i)), 22050, (x * 32767).astype(np.int16))
            f.write("LJ%03d|%s|%s\n" % (i, t, t))
    rows = preprocess.build_from_path(str(in_dir), str(out_b), num_workers=2, batch_clips=3)
    rows_ref = [(a, b, int(n), t) for a, b, n, t in DROPIN["ljspeech"]["out"]["rows"].tolist()]
    assert rows == rows_ref and len(rows) == 4
    kept = [i for i, t in enumerate(texts) if len(t) >= hp["min_text"]]
    for i, (spec_name, mel_name, n_frames, _) in zip(kept, rows):
        wav = audio.load_wav(str(in_dir / "wavs" / ("LJ%03d.wav" % i)))
        a, b = audio.spectrogram(wav).astype(np.float32).T, np.load(out_b / spec_name)
        assert a.shape == (n_frames, 513) and b.dtype == np.float32 and np.array_equal(a, b)
        a, b = audio.melspectrogram(wav).astype(np.float32).T, np.load(out_b / mel_name)
        assert a.shape == (n_frames, 80) and np.array_equal(a, b)
    frames, hours = preprocess.write_metadata(rows, str(out_b))
    lines = open(out_b / "train.txt", encoding="utf-8").read().splitlines()
    assert len(lines) == 4 and lines[0].split("|")[:3] == ["ljspeech-spec-00001.npy", "ljspeech-mel-00001.npy",
                                                           str(rows[0][2])] and frames == sum(r[2] for r in rows)
    # and against the numpy restatement of audio.py for one utterance
    ref_lin, ref_mel = A.process_utterance(audio.load_wav(str(in_dir / "wavs" / "LJ000.wav")))
    got = np.load(out_b / rows[0][0])
    assert got.shape == ref_lin.shape and np.abs(got - ref_lin).mean() < 2e-4
