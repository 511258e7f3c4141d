#!/usr/bin/env python
"""Golden vectors for the loss / batching code of the reference's ``train.py``, produced by EXECUTING that file
(unchanged, through oracle/ref_harness.py, which only stands in for uninstalled logging / CLI / text packages).

    python tests/golden/make_train_golden.py          (build container: needs /root/reference)

Writes tests/golden/train_fns.*.npz:

* ``mask*``      ``sequence_mask`` (train.py:261-271)
* ``specloss*``  ``spec_loss`` (train.py:547-582) incl. the priority-bin branch (:559-567) and w = 0 / bw = 0 corners
* ``guided*``    ``guided_attentions`` (train.py:585-601)
* ``collate*``   ``collate_fn`` (train.py:293-360), single- and multi-speaker, r/downsample_step variants
* ``step*``      the INLINE loss code of ``train()`` (train.py:665-740): ``train()`` itself is run for one step on a
                 stand-in model that returns fixed leaf tensors, so the total loss and its gradient w.r.t. every model
                 output are the reference's own (clip_thresh = 0, optimizer lr = 0).
"""
import os
import sys
import warnings

import numpy as np
import torch
from torch import nn

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_harness as H  # noqa: E402
import golden_util as G  # noqa: E402

OUT = {}


def put(case, group, name, value):
    OUT["%s|%s|%s" % (case, group, name)] = value.detach().cpu().numpy() if torch.is_tensor(value) else np.asarray(value)


class FixedOutputs(nn.Module):
    """Stand-in model for train(): returns stored leaves, so d(loss)/d(outputs) lands in their .grad."""

    def __init__(self, mel, lin, attn, done, linear_dim):
        super().__init__()
        self.mel, self.lin = nn.Parameter(mel), nn.Parameter(lin)
        self.attn, self.done = nn.Parameter(attn), nn.Parameter(done)
        self.linear_dim = linear_dim

    def get_trainable_parameters(self):
        return self.parameters()

    def forward(self, x, mel, speaker_ids=None, text_positions=None, frame_positions=None, input_lengths=None):
        return self.mel, self.lin, self.attn, self.done


def main():
    tr = H.load_train("reference")
    hp = tr.hparams
    gen = torch.Generator().manual_seed(0)

    # ---- sequence_mask -------------------------------------------------------------------------------
    lengths = torch.tensor([5, 0, 9, 3])
    put("mask0", "in", "lengths", lengths)
    put("mask0", "out", "0", tr.sequence_mask(lengths, max_len=9))
    put("mask1", "in", "lengths", lengths)
    put("mask1", "out", "0", tr.sequence_mask(lengths))           # max_len=None branch

    # ---- spec_loss -----------------------------------------------------------------------------------
    cases = [("specloss0", 0.5, 0.1, None, 0.0), ("specloss1", 0.5, 0.1, 70, 0.3), ("specloss2", 0.0, 0.1, 70, 0.5),
             ("specloss3", 0.5, 0.0, None, 0.0), ("specloss4", 1.0, 0.3, 200, 1.0)]
    for name, w, bw, pbin, pw in cases:
        hp.set_hparam("masked_loss_weight", w)
        hp.set_hparam("binary_divergence_weight", bw)
        B, T, D = 3, 17, 257
        y_hat = torch.rand(B, T, D, generator=gen).clamp(1e-3, 1 - 1e-3).requires_grad_(True)
        y = torch.rand(B, T, D, generator=gen)
        lens = torch.tensor([17, 9, 13])
        mask = tr.sequence_mask(lens, max_len=T).unsqueeze(-1) if w > 0 else None
        l1, bd = tr.spec_loss(y_hat, y, mask, priority_bin=pbin, priority_w=pw)
        ((1 - bw) * l1 + bw * bd.sum()).backward()
        put(name, "in", "y_hat", y_hat)
        put(name, "in", "y", y)
        put(name, "in", "lengths", lens)
        put(name, "meta", "cfg", np.array([w, bw, -1 if pbin is None else pbin, pw], dtype=np.float64))
        put(name, "out", "l1", l1)
        put(name, "out", "bd", bd.reshape(()))
        put(name, "out", "grad", y_hat.grad)

    # ---- guided_attentions ---------------------------------------------------------------------------
    il, tl = np.array([7, 12, 3]), np.array([10, 4, 9])
    for name, g in (("guided0", 0.2), ("guided1", 0.4)):
        put(name, "in", "input_lengths", il)
        put(name, "in", "target_lengths", tl)
        put(name, "meta", "g", np.float64(g))
        put(name, "out", "0", tr.guided_attentions(il, tl, 11, g=g))

    # ---- collate_fn ----------------------------------------------------------------------------------
    for name, r, ds, nspk in (("collate0", 1, 4, 1), ("collate1", 1, 4, 5), ("collate2", 2, 1, 1), ("collate3", 3, 4, 1)):
        hp.set_hparam("outputs_per_step", r)
        hp.set_hparam("downsample_step", ds)
        utts = H.synthetic_utterances(4, seed=11 + r, n_speakers=nspk, min_frames=24, max_frames=61, linear_dim=33,
                                      mel_dim=8)
        x, ilen, mel, y, (tpos, fpos), done, tlen, spk = tr.collate_fn(utts)
        put(name, "meta", "cfg", np.array([r, ds, nspk]))
        for i, u in enumerate(utts):
            put(name, "in", "text%d" % i, u[0])
            put(name, "in", "mel%d" % i, u[1])
            put(name, "in", "lin%d" % i, u[2])
            if nspk > 1:
                put(name, "in", "spk%d" % i, np.int64(u[3]))
        for k, v in (("x", x), ("input_lengths", ilen), ("mel", mel), ("y", y), ("text_positions", tpos),
                     ("frame_positions", fpos), ("done", done), ("target_lengths", tlen)):
            put(name, "out", k, v)
        if spk is not None:
            put(name, "out", "speaker_ids", spk)

    # ---- the inline loss of train() ------------------------------------------------------------------
    for name, w, bw, pw, guided, nspk in (("step0", 0.5, 0.1, 0.0, True, 1), ("step1", 0.5, 0.1, 0.25, True, 3),
                                           ("step2", 0.0, 0.0, 0.0, False, 1)):
        H.apply_preset(tr, "deepvoice3_ljspeech", masked_loss_weight=w, binary_divergence_weight=bw,
                       priority_freq_weight=pw, use_guided_attention=guided,
                       eval_interval=10 ** 9)
        r, ds = hp.outputs_per_step, hp.downsample_step
        utts = H.synthetic_utterances(3, seed=21, n_speakers=nspk, min_text=9, max_text=20, min_frames=40,
                                      max_frames=77)
        batch = tr.collate_fn(utts)
        x, ilen, mel, y, (tpos, fpos), done, tlen, spk = batch
        B, T_lin, T_dec, Ts = x.size(0), y.size(1), y.size(1) // ds // r, x.size(1)
        outs = (torch.rand(B, T_dec, 80, generator=gen).clamp(1e-3, 1 - 1e-3),
                torch.rand(B, T_lin, 513, generator=gen).clamp(1e-3, 1 - 1e-3),
                torch.softmax(2 * torch.randn(2, B, T_dec, Ts, generator=gen), -1),
                torch.rand(B, T_dec, 1, generator=gen).clamp(1e-3, 1 - 1e-3))
        model = FixedOutputs(*outs, linear_dim=513)
        writer = H.ScalarLog()
        opt = torch.optim.SGD(model.parameters(), lr=0.0)
        tr.global_step, tr.global_epoch = 0, 0
        tr.train(torch.device("cpu"), model, [batch], opt, writer, init_lr=0.0, checkpoint_dir="/tmp",
                 checkpoint_interval=10 ** 9, nepochs=1, clip_thresh=0)
        put(name, "meta", "cfg", np.array([w, bw, pw, float(guided), hp.priority_freq, hp.sample_rate,
                                           hp.guided_attention_sigma, r, ds], dtype=np.float64))
        for k, v in (("x", x), ("input_lengths", ilen), ("mel", mel), ("y", y), ("done", done),
                     ("target_lengths", tlen)):
            put(name, "in", k, v)
        for k, v in zip(("mel_out", "lin_out", "attn", "done_hat"), outs):
            put(name, "in", k, v)
        for tag, vals in writer.scalars.items():
            put(name, "out", tag.replace(" ", "_"), np.float64(vals[0][1]))
        for k, p in (("mel_out", model.mel), ("lin_out", model.lin), ("attn", model.attn), ("done_hat", model.done)):
            put(name, "out", "grad_" + k, p.grad if p.grad is not None else torch.zeros_like(p))

    G.save("train_fns.npz", OUT)


if __name__ == "__main__":
    main()
