#!/usr/bin/env python
"""Golden vectors for tests/test_dropin.py, produced by EXECUTING the reference's own ``train.py``, ``synthesis.py``
and ``ljspeech.py`` on the reference package, on the CPU (through oracle/ref_harness.py, which only stands in for
uninstalled logging / CLI / text packages).  Needs oracle/_ref (``python oracle/make_ref.py``).

    python tests/golden/make_dropin_golden.py

Writes tests/golden/dropin.*.npz:

* ``<preset>|meta|hparams``   the reference's hparams after ``presets/<preset>.json`` (train.py:936-939), as JSON
* ``build_model``             ``build_model()`` (train.py:812-840) of deepvoice3_ljspeech under seed 0: state_dict keys,
                              shapes and the SHA-256 of every tensor's bytes
* ``train_<preset>``          the scalars ``train()`` logs over 4 optimizer steps (dropout 0) on synthetic utterances
* ``tts``                     ``synthesis.tts()`` of "hello b200": alignment, linear spectrogram, mel, waveform length
* ``ljspeech``                the ``train.txt`` rows ``ljspeech._process_utterance`` returns for five synthetic clips
"""
import hashlib
import json
import os
import sys
import tempfile
import types
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from oracle import audio_oracle as A  # noqa: E402
from oracle import ref_harness as H  # noqa: E402
import golden_util as G  # noqa: E402

PRESETS = (("deepvoice3_ljspeech", 1), ("nyanko_ljspeech", 1), ("deepvoice3_vctk", 108))
TAGS = ("loss", "mel_l1_loss", "linear_l1_loss", "done_loss", "attn_loss", "gradient norm")
# what tests/test_dropin.py feeds both sides
TRAIN_UTTS = dict(n=16, seed=3, min_text=40, max_text=100, min_frames=200, max_frames=400)
TTS_TEXT, TTS_STEPS = "hello b200", 24
LJ_LENS = [30001, 22050, 5000, 47777, 12345]
OUT = {}


def put(case, group, name, value):
    OUT["%s|%s|%s" % (case, group, name)] = value.detach().cpu().numpy() if torch.is_tensor(value) else np.asarray(value)


def lj_texts():
    texts = ["the quick brown fox jumps over the lazy dog %d" % i for i in range(len(LJ_LENS))]
    texts[2] = "too short"                                  # < hparams.min_text = 20: skipped
    return texts


def hparams_and_build_model():
    for preset, _ in PRESETS:
        tr = H.load_train("reference")
        hp = H.apply_preset(tr, preset)
        put(preset, "meta", "hparams", json.dumps(hp.values(), sort_keys=True))
    tr = H.load_train("reference")
    H.apply_preset(tr, "deepvoice3_ljspeech")
    torch.manual_seed(0)
    sd = tr.build_model().state_dict()
    put("build_model", "meta", "keys", np.array(list(sd.keys())))
    put("build_model", "meta", "shapes", np.array([str(tuple(v.shape)) for v in sd.values()]))
    put("build_model", "out", "sha256", np.array([hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest()
                                                  for v in sd.values()]))


def train_loops():
    from torch.utils.data import DataLoader
    for preset, n_speakers in PRESETS:
        tr = H.load_train("reference")
        hp = H.apply_preset(tr, preset, dropout=0.0, eval_interval=10 ** 9)
        torch.manual_seed(0)
        model = tr.build_model()
        opt = torch.optim.Adam(model.get_trainable_parameters(), lr=hp.initial_learning_rate,
                               betas=(hp.adam_beta1, hp.adam_beta2), eps=hp.adam_eps,
                               weight_decay=hp.weight_decay, amsgrad=hp.amsgrad)
        utts = H.synthetic_utterances(TRAIN_UTTS["n"], seed=TRAIN_UTTS["seed"], n_speakers=n_speakers,
                                      min_text=TRAIN_UTTS["min_text"], max_text=TRAIN_UTTS["max_text"],
                                      min_frames=TRAIN_UTTS["min_frames"], max_frames=TRAIN_UTTS["max_frames"])
        loader = DataLoader(utts, batch_size=4, collate_fn=tr.collate_fn, shuffle=False)
        writer = H.ScalarLog()
        tr.global_step, tr.global_epoch = 0, 0
        with tempfile.TemporaryDirectory() as tmp:
            tr.train(torch.device("cpu"), model, loader, opt, writer, init_lr=hp.initial_learning_rate,
                     checkpoint_dir=tmp, checkpoint_interval=10 ** 9, nepochs=1, clip_thresh=hp.clip_thresh)
        for tag in TAGS:
            put("train_" + preset, "out", tag.replace(" ", "_"), np.array([v for _, v in writer.scalars[tag]]))
        print(preset, {t: writer.scalars[t][0][1] for t in TAGS})


def tts():
    shim = types.ModuleType("audio")                       # lws is not installed: numpy restatement of audio.py
    shim._denormalize = lambda S: np.clip(S, 0, 1) * 100.0 - 100.0
    shim.inv_spectrogram = lambda S: A.inv_spectrogram(S, n_iter=4)
    syn = H.load_synthesis("reference", shim)
    tr = H.load_train("reference")
    H.apply_preset(tr, "deepvoice3_ljspeech")
    torch.manual_seed(0)
    model = tr.build_model()
    sd = model.state_dict()
    sd["seq2seq.decoder.fc.bias"] = torch.full_like(sd["seq2seq.decoder.fc.bias"], -8.0)   # never "done"
    model.load_state_dict(sd)
    model.seq2seq.decoder.max_decoder_steps = TTS_STEPS
    waveform, alignment, spectrogram, mel = syn.tts(model, TTS_TEXT, p=0, speaker_id=None, fast=True)
    put("tts", "out", "alignment", alignment)
    put("tts", "out", "spectrogram", spectrogram)
    put("tts", "out", "mel", mel)
    put("tts", "meta", "waveform_len", np.int64(len(waveform)))


def ljspeech():
    from scipy.io import wavfile
    shim = types.ModuleType("audio")                       # CPU restatement: only the rows are stored
    shim.load_wav = lambda p: wavfile.read(p)[1].astype(np.float32) / 32768.0
    shim.spectrogram = lambda y: A.spectrogram(y)
    shim.melspectrogram = lambda y: A.melspectrogram(y)
    lj = H.load_ljspeech(shim)
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        for i, (n, t) in enumerate(zip(LJ_LENS, lj_texts())):
            if len(t) < lj.hparams.min_text:
                continue
            path = os.path.join(tmp, "LJ%03d.wav" % i)
            wavfile.write(path, 22050, (A.synthetic_clip(70 + i, n=n) * 32767).astype(np.int16))
            rows.append(lj._process_utterance(tmp, len(rows) + 1, path, t))
    put("ljspeech", "out", "rows", np.array([[str(c) for c in r] for r in rows]))


if __name__ == "__main__":
    torch.set_num_threads(min(os.cpu_count() or 8, 16))
    hparams_and_build_model()
    tts()
    ljspeech()
    train_loops()
    G.save("dropin.npz", OUT)
