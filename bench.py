#!/usr/bin/env python
"""Headline benchmark: mel-frames/sec of one training step (B=16 per GPU, T_text=128, T_mel=800) of the
deepvoice3_ljspeech preset on synthetic data, plus the fused-ConvBlock roofline and the CPU baseline.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \\
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU arm: the UNMODIFIED reference package + the reference's own
                                              # train.py loop (oracle/_ref), on the host cores

One step = zero_grad -> forward -> the reference's losses (train.py:704-740) -> backward -> (NCCL gradient
all-reduce) -> clip_grad_norm(0.1) -> Adam.  Timed with CUDA events on the launching stream, barrier +
synchronize on both sides, max over ranks.  A step touches > 1.5 GB of weights, optimizer state and
activations, i.e. far more than the 126 MB L2 ("inputs larger than L2").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PRESETS = {
    # train.py:812-840 hparams -> builder kwargs, values from presets/*.json
    "deepvoice3_ljspeech": ("deepvoice3", dict(
        n_speakers=1, speaker_embed_dim=16, n_vocab=149, embed_dim=256, mel_dim=80, linear_dim=513, r=1,
        downsample_step=4, padding_idx=0, dropout=0.05, kernel_size=3, encoder_channels=512,
        decoder_channels=256, converter_channels=256, use_memory_mask=True,
        trainable_positional_encodings=False, force_monotonic_attention=True,
        use_decoder_state_for_postnet_input=True, max_positions=512, speaker_embedding_weight_std=0.01,
        freeze_embedding=False, window_ahead=3, window_backward=1, key_projection=True,
        value_projection=True), dict(guided_attention_sigma=0.2)),
    "nyanko_ljspeech": ("nyanko", dict(
        n_speakers=1, speaker_embed_dim=16, n_vocab=149, embed_dim=128, mel_dim=80, linear_dim=513, r=1,
        downsample_step=4, padding_idx=0, dropout=0.05, kernel_size=3, encoder_channels=256,
        decoder_channels=256, converter_channels=256, use_memory_mask=True,
        trainable_positional_encodings=False, force_monotonic_attention=True,
        use_decoder_state_for_postnet_input=True, max_positions=512, speaker_embedding_weight_std=0.01,
        freeze_embedding=False, window_ahead=3, window_backward=1, key_projection=False,
        value_projection=False), dict(guided_attention_sigma=0.2)),
    "deepvoice3_vctk": ("deepvoice3_multispeaker", dict(
        n_speakers=108, speaker_embed_dim=16, n_vocab=149, embed_dim=256, mel_dim=80, linear_dim=513, r=1,
        downsample_step=4, padding_idx=0, dropout=0.05, kernel_size=3, encoder_channels=512,
        decoder_channels=256, converter_channels=256, use_memory_mask=True,
        trainable_positional_encodings=False, force_monotonic_attention=True,
        use_decoder_state_for_postnet_input=True, max_positions=1024, speaker_embedding_weight_std=0.05,
        freeze_embedding=False, window_ahead=3, window_backward=1, key_projection=True,
        value_projection=True), dict(guided_attention_sigma=0.4)),
}
B, T_TEXT, T_MEL = 16, 128, 800
METRIC = "mel-frames/sec training step (B=16,T_mel=800)"
WORKLOAD = "%s training step, B=16/GPU, T_text=128, T_mel=800 (T_dec=200)"
NCU_TRAFFIC_GATED_512_800 = 90.40e6   # dram__bytes_read.sum + dram__bytes_write.sum (58.82 + 31.58 MB) of the (16,512,800)
                                      # gated forward, profiles/r02_ncu_full_conv.csv (`ncu --set full` of this kernel)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"],
                                   r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}



def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# -------------------------------------------------------------------------------------------------
# The reference itself: oracle/_ref (an unmodified copy of the reference package + train.py, oracle/make_ref.py) driven
# through the reference's own train() loop (train.py:604-785) on reference collate_fn batches.  Used for
#   * the CPU arm (`--impl reference`, `cpu_baseline`): device = cpu, all the host threads oneDNN scales to;
#   * `gpu_eager_baseline`: the same modules in PyTorch eager on the B200 (cuDNN / cuBLAS), TF32 off and on -- the
#     honest GPU competitor of SURVEY.md section 8(d).
# -------------------------------------------------------------------------------------------------
class _TimedLoader:
    """Yields the same host batch n times and records when each step starts (= when the previous one finished:
    train() ends every step with .item() reads, so the stream is drained)."""

    def __init__(self, batch, n, cuda):
        self.batch, self.n, self.cuda, self.t = batch, n, cuda, []

    def _stamp(self):
        if self.cuda:
            torch.cuda.synchronize()
        self.t.append(time.perf_counter())

    def __len__(self):
        return self.n

    def __iter__(self):
        for _ in range(self.n):
            self._stamp()
            yield self.batch
        self._stamp()


def reference_train_throughput(preset, device, steps, warmup, threads=None, tf32=False, budget_s=None):
    """-> (mel-frames/s, seconds per step (median), steps timed).  None if oracle/_ref is not available."""
    from oracle import ref_harness as H
    if H.ref_root() is None:
        return None
    import tempfile
    if device.type == "cpu":
        # oneDNN's small convolutions stop scaling (and on shared 100+-core hosts collapse) beyond a few dozen
        # threads: use at most 32 (measured: 128 threads on the B200 host = 134 s/step vs ~1-6 s/step at 8-32).
        torch.set_num_threads(threads or min(os.cpu_count() or 8, 32))
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    try:
        tr = H.load_train("reference")
        hp = H.apply_preset(tr, preset, eval_interval=10 ** 9)
        n_spk = hp.n_speakers
        rng = np.random.RandomState(1234)
        # B utterances of exactly T_TEXT characters and T_MEL - 4 frames: collate_fn (train.py:293-360) adds the
        # r * downsample_step = 4 leading zero frames -> T_mel = 800, T_dec = 200
        utts = []
        for _ in range(B):
            u = (rng.randint(2, 149, T_TEXT).astype(np.int64), rng.rand(T_MEL - 4, 80).astype(np.float32),
                 rng.rand(T_MEL - 4, 513).astype(np.float32))
            utts.append(u + (int(rng.randint(0, n_spk)),) if n_spk > 1 else u)
        batch = tr.collate_fn(utts)
        assert batch[2].shape[1] == T_MEL and batch[0].shape[1] == T_TEXT
        torch.manual_seed(1234)
        model = tr.build_model().to(device)
        opt = torch.optim.Adam(model.get_trainable_parameters(), lr=hp.initial_learning_rate,
                               betas=(hp.adam_beta1, hp.adam_beta2), eps=hp.adam_eps, weight_decay=hp.weight_decay,
                               amsgrad=hp.amsgrad)
        n = warmup + steps
        if budget_s is not None:                      # bounded sample: time one step first
            probe = _TimedLoader(batch, 1, device.type == "cuda")
            tr.global_step, tr.global_epoch = 0, 0
            with tempfile.TemporaryDirectory() as tmp, open(os.devnull, "w") as null:
                _quiet(lambda: tr.train(device, model, probe, opt, H.ScalarLog(), init_lr=hp.initial_learning_rate,
                                        checkpoint_dir=tmp, checkpoint_interval=10 ** 9, nepochs=1,
                                        clip_thresh=hp.clip_thresh), null)
            one = probe.t[1] - probe.t[0]
            n = max(2, min(n, int(budget_s / max(one, 1e-3))))
            warmup = min(warmup, n - 1) if n > 1 else 0
        loader = _TimedLoader(batch, n, device.type == "cuda")
        tr.global_step, tr.global_epoch = 0, 0
        with tempfile.TemporaryDirectory() as tmp, open(os.devnull, "w") as null:
            _quiet(lambda: tr.train(device, model, loader, opt, H.ScalarLog(), init_lr=hp.initial_learning_rate,
                                    checkpoint_dir=tmp, checkpoint_interval=10 ** 9, nepochs=1,
                                    clip_thresh=hp.clip_thresh), null)
        dt = np.diff(np.array(loader.t))[warmup:]
        sec = float(np.median(dt))
        del model, opt
        if device.type == "cuda":
            torch.cuda.empty_cache()
        return B * T_MEL / sec, sec, len(dt)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _quiet(fn, null):
    """train.py prints / tqdm-writes progress: keep stdout a single JSON line."""
    import contextlib
    import warnings
    with contextlib.redirect_stdout(null), contextlib.redirect_stderr(null), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn()


def cpu_port_throughput(preset, steps, warmup, threads=None):
    """Fallback CPU arm when oracle/_ref is absent: the oracle PORT of the reference modules + losses (kind "port")."""
    from oracle import dv3_oracle as O
    from oracle.specs import spec_from_builder
    from deepvoice3_pytorch_b200 import builder
    from deepvoice3_pytorch_b200.train_step import make_synthetic_batch, noam_learning_rate_decay
    threads = threads or min(os.cpu_count() or 8, 32)
    torch.set_num_threads(threads)
    bname, kw, extra = PRESETS[preset]
    torch.manual_seed(1234)
    model = getattr(builder, bname)(**kw)                 # parameter container only; never run on the CPU
    spec = spec_from_builder(bname, **dict(kw, dropout=0.0))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    frozen = {"seq2seq.decoder.embed_query_positions.weight", "seq2seq.decoder.embed_keys_positions.weight"}
    leaves = [v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and k not in frozen]
    opt = torch.optim.Adam(leaves, lr=5e-4, betas=(0.5, 0.9), eps=1e-6)
    b = make_synthetic_batch(B, T_TEXT, T_MEL, n_speakers=kw["n_speakers"])
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        for g in opt.param_groups:
            g["lr"] = noam_learning_rate_decay(5e-4, i)
        opt.zero_grad()
        outs = O.model_forward(sd, spec, b["x"], b["mel"], b.get("speaker_ids"), b["text_positions"],
                               b["frame_positions"], b["input_lengths"])
        loss = O.training_loss(outs, b["mel"], b["y"], b["done"], b["input_lengths"],
                               b["target_lengths"].numpy(), guided_sigma=extra["guided_attention_sigma"])
        loss.backward()
        torch.nn.utils.clip_grad_norm_(leaves, 0.1)
        opt.step()
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
            if sum(ts) > 60.0:
                break
    sec = float(np.median(ts))
    return B * T_MEL / sec, sec, len(ts)


def cpu_arm(preset, steps, warmup, budget_s=None):
    """-> dict(value, sec, cores, kind, n) for the CPU baseline."""
    cores = min(os.cpu_count() or 8, 32)
    r = reference_train_throughput(preset, torch.device("cpu"), steps, warmup, threads=cores, budget_s=budget_s)
    kind = "reference"
    if r is None:
        r, kind = cpu_port_throughput(preset, steps, warmup, threads=cores), "port"
    return {"value": r[0], "sec": r[1], "cores": cores, "kind": kind, "n": r[2]}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = min(args.steps, 5), min(args.warmup, 1)
    c = cpu_arm(args.preset, steps, warmup)
    how = ("the UNMODIFIED reference package + reference train.py train() loop (oracle/_ref), dropout on, PyTorch CPU"
           if c["kind"] == "reference" else "oracle port of the reference (oracle/_ref missing)")
    sample = "%d full steps (B=16,T_text=128,T_mel=800) after %d warm-up, median; %s; %s" % (c["n"], warmup, how,
                                                                                             cpu_model())
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": c["value"], "unit": "mel-frames/s", "n_gpus": args.gpus,
        "steps": c["n"], "warmup": warmup, "ms_per_step": c["sec"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % args.preset},
        "cpu_baseline": {"value": c["value"], "unit": "mel-frames/s", "cores": c["cores"], "kind": c["kind"],
                         "sample": sample, "cpu": cpu_model()},
        "e2e": {"value": c["value"], "unit": "mel-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# -------------------------------------------------------------------------------------------------
# GPU arm
# -------------------------------------------------------------------------------------------------
def _time_launch(launch, flush, reps=10):
    for _ in range(3):
        launch()
    ts = []
    for _ in range(reps):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); launch(); e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) * 1e-3)
    return float(np.mean(ts))


def convblock_roofline(dev, pk, pk_kind):
    """The time-dominant kernel FAMILY of the step: tc_conv_kernel (tcgen05 gated forward / conv / data-gradient GEMM;
    42 % of the GPU time of a step, profiles/r02_step_profile.txt).  Every ConvBlock shape of the ljspeech model is
    timed -- gated forward and data gradient, operands prepared outside, CUDA events on the launching stream, L2
    flushed between launches -- and aggregated with the number of such launches per training step:
        achieved = sum_i n_i * flops_i / sum_i n_i * t_i      (ALGORITHMIC flops: 2*B*T*2C*C*k per launch)
    next to the largest member (B=16, C=512, T=800, k=3) on its own, and BASELINE.json's "ConvBlock HBM GB/s" view
    (algorithmic bytes 4*[2*B*C*T + 2C*C*k + 4C] per forward launch, BASELINE.md section 4)."""
    from deepvoice3_pytorch_b200 import ops
    assert ops.conv_math in ("tc", "bf16x3")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    bf, f16 = torch.bfloat16, torch.float16
    # (C, T, launches per step of each of {gated forward, data gradient}) for deepvoice3_ljspeech, B = 16, k = 3
    shapes = [(512, 128, 10), (256, 200, 7), (256, 400, 2), (256, 800, 4), (512, 800, 2)]
    Bc, k, d = 16, 3, 1
    rows, big = [], None
    for C, T, n in shapes:
        v = torch.randn(2 * C, C, k, device=dev) * (4.0 / (k * C)) ** 0.5
        g = v.pow(2).sum((1, 2), keepdim=True).sqrt()
        bias = torch.zeros(2 * C, device=dev)
        x = torch.randn(Bc, C, T, device=dev)
        y, sa, ss = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
        inv, scale = torch.empty(2 * C, device=dev), torch.empty(2 * C, device=dev)
        wfwd = torch.empty(2, k, 2 * C, C, device=dev, dtype=f16)
        wbwd = torch.empty(2, k, C, 2 * C, device=dev, dtype=bf)
        ops.lib.call("dv3_tc_weightnorm_fwd", ops._p(v), ops._p(g), ops._p(inv), ops._p(scale), ops._p(wfwd), 2,
                     ops._p(wbwd), 2 * C, C, k, ops._stream())
        xs = torch.empty(2, Bc, T, C, device=dev, dtype=f16)
        ops.lib.call("dv3_tc_split_input", ops._p(x), ops._p(xs), 2, None, Bc, C, T, k, d, 0, 0.0, None, 0,
                     ops._stream())
        dab = torch.empty(2, Bc, T, 2 * C, device=dev, dtype=bf)
        ops.lib.call("dv3_tc_gate_bwd_split", ops._p(x), ops._p(sa.normal_()), ops._p(ss.uniform_()), None, ops._p(dab),
                     None, None, Bc, C, T, 0, 1, ops._stream())
        dx = torch.empty_like(x)

        def fwd():
            ops.lib.call("dv3_tc_convblock_fwd", ops._p(xs), ops._p(wfwd), 2, ops._p(bias), None, ops._p(x), ops._p(y),
                         ops._p(sa), ops._p(ss), Bc, C, T, k, d, 0, 0, 1, None, ops._stream())

        def dgrad():
            ops.lib.call("dv3_tc_conv", ops._p(dab), ops._p(wbwd), 2, ops._p(dx), Bc, 2 * C, C, T, k, d, 0, 1, None, 0,
                         0.0, None, 0, 1, ops._p(y), None, 0.7071067811865476, None, ops._stream())
        tf, tb = _time_launch(fwd, flush), _time_launch(dgrad, flush)
        flops = 2.0 * Bc * T * 2 * C * C * k
        rows.append({"B": Bc, "C": C, "T": T, "k": k, "launches_per_step": n, "fwd_us": tf * 1e6, "dgrad_us": tb * 1e6,
                     "fwd_tflops": flops / tf / 1e12, "dgrad_tflops": flops / tb / 1e12})
        if (C, T) == (512, 800):
            big = (tf, flops, 4.0 * (2 * Bc * C * T + 2 * C * C * k + 4 * C))
    tot_f = sum(r["launches_per_step"] * 2 * 2.0 * r["B"] * r["T"] * 2 * r["C"] * r["C"] * r["k"] for r in rows)
    tot_t = sum(r["launches_per_step"] * (r["fwd_us"] + r["dgrad_us"]) * 1e-6 for r in rows)
    ach = tot_f / tot_t / 1e12
    tf, flops, alg_bytes = big
    return {
        "bound": "tensor",
        "kernel": "tc_conv_kernel family (persistent tcgen05 gated-forward / data-gradient GEMMs of all 25 ConvBlocks "
                  "of the step: 50 launches, time-weighted) via dv3_tc_convblock_fwd / dv3_tc_conv",
        "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
        "issued_tflops": 3 * ach, "issued_frac": 3 * ach / pk["bf16_tflops"],
        "note": "achieved counts ALGORITHMIC flops (one fp32 multiply-add per term); the kernels issue 3 fp16 MMA "
                "passes per term (hi*hi, hi*lo, lo*hi of fp16 operand pairs) for fp32-class results",
        "family_us_per_step": tot_t * 1e6, "shapes": rows, "peak_source": pk_kind,
        # dram__bytes_read.sum + dram__bytes_write.sum of the (16,512,800) gated forward from the committed
        # `ncu --set full` capture of THIS kernel (profiles/r02_ncu_full_conv.csv)
        "traffic": NCU_TRAFFIC_GATED_512_800,
        "largest_member": {"shape": "(B=16,C=512,T=800,k=3) gated forward", "launch_us": tf * 1e6,
                           "achieved": flops / tf / 1e12, "frac": flops / tf / 1e12 / pk["bf16_tflops"],
                           "alg_flops": flops},
        "hbm": {"bound": "hbm", "achieved": alg_bytes / tf / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": alg_bytes / tf / 1e9 / pk["hbm_gbs"], "alg_bytes": alg_bytes,
                "note": "BASELINE.json's 'ConvBlock HBM GB/s' for the largest member: algorithmic bytes / launch time; the "
                        "block is a dense contraction (686 FLOP/B here), so this roof does not bind"},
    }


def run_gpu_arm(args):
    import torch.distributed as dist
    from deepvoice3_pytorch_b200 import builder, ops
    from deepvoice3_pytorch_b200._lib import lib
    from deepvoice3_pytorch_b200.train_step import TrainStep, make_synthetic_batch, to_device

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback; --impl reference is the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run_step, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            run_step()
        e.record()
        barrier()
        t = torch.tensor([s.elapsed_time(e) * 1e-3], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def make_step(preset, math, graph=True):
        ops.conv_math = math
        bname, kw, extra = PRESETS[preset]
        torch.manual_seed(1234)                  # same initial weights everywhere (TrainStep also broadcasts rank 0's)
        model = getattr(builder, bname)(**kw).to(dev)
        st = TrainStep(model, use_graph=graph, **extra)
        host_b = make_synthetic_batch(B, T_TEXT, T_MEL, n_speakers=kw["n_speakers"], seed=1234 + rank, pin=True)
        return st, host_b

    ops.conv_math = args.math
    step, host = make_step(args.preset, args.math, graph=not args.no_graph)
    ops.rng.manual_seed(1234 + rank, dev)
    resident = to_device(host, dev)

    # ---- device-resident throughput (value) ------------------------------------------------------
    # nvidia-smi needs ~0.5 s to deliver its first sample and a 20-step timed region lasts ~0.1 s, so the sampler
    # runs from the warm-up to the end of the e2e region (the GPU is under the same load throughout).
    clocks = ClockSampler(local).__enter__()
    for _ in range(max(args.warmup, 3)):
        loss = step.step(resident)
    torch.cuda.synchronize()
    ops.check_index_errors()
    l0 = lib.raw("dv3_launch_count")()
    last = {}

    def timed_step():
        last["loss"] = step.step(resident)
    t_res = timed(timed_step, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["loss"], step.model)
    launches = (lib.raw("dv3_launch_count")() - l0) // args.steps
    if step.launches_per_step is not None:       # graph replay: the launches were recorded at capture time
        launches = step.launches_per_step
    loss_val = float(loss.item())
    assert np.isfinite(loss_val), "training diverged"

    # ---- end to end: pinned host batch -> H2D every step, loss read back every step ------------------
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))
    sink = []
    # Every step uploads its own batch from pinned host memory and reads the loss back.  The upload of step i+1 is
    # issued on a copy stream before step i is launched (what a pinned-memory DataLoader with non_blocking copies
    # does), so the PCIe transfer overlaps the previous step's compute; both are inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)

    def upload():
        with torch.cuda.stream(copy_stream):
            b = to_device(host, dev)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, ev

    pending = [upload()]
    # The loss of step i is copied into pinned host memory on the compute stream right after the step and READ by the
    # host while step i+1 runs (one step of lag, what an asynchronous logger does): every step's result still crosses
    # PCIe and is consumed inside the timed region, but the host never idles the GPU while it prepares the next step.
    loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    inflight = []

    def read_back():
        slot = inflight.pop(0)
        loss_ev[slot].synchronize()
        sink.append(float(loss_host[slot]))               # D2H result of an earlier step

    def e2e_step():
        batch, ev = pending.pop()
        torch.cuda.current_stream().wait_event(ev)
        pending.append(upload())                          # prefetch the next step's batch
        loss_t = step.step(batch)
        for v in batch.values():                          # the buffers were produced on the copy stream
            if torch.is_tensor(v):
                v.record_stream(torch.cuda.current_stream())
        slot = step.global_step & 1
        loss_host[slot].copy_(loss_t.detach().reshape(()), non_blocking=True)
        loss_ev[slot].record()
        inflight.append(slot)
        if len(inflight) > 1:
            read_back()                                   # the previous step's loss (its copy finished long ago)
    for _ in range(2):
        e2e_step()

    def e2e_region():
        for _ in range(args.steps):
            e2e_step()
        while inflight:                                   # the last step's loss is read inside the timed region too
            read_back()
    n_before = len(sink)
    barrier()
    s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s_ev.record()
    e2e_region()
    e_ev.record()
    barrier()
    t_loc = torch.tensor([s_ev.elapsed_time(e_ev) * 1e-3], device=dev)
    if world > 1:
        dist.all_reduce(t_loc, op=dist.ReduceOp.MAX)
    t_e2e = float(t_loc.item())
    assert len(sink) - n_before >= args.steps and all(np.isfinite(v) for v in sink), "e2e: every step's loss is read"
    t_extra = time.perf_counter()
    while len(clocks.rows) < 3 and time.perf_counter() - t_extra < 3.0:      # keep the load on until sampled
        step.step(resident)
    torch.cuda.synchronize()
    clocks.__exit__()

    frames = B * T_MEL * world
    out = {
        "metric": METRIC, "value": frames * args.steps / t_res, "unit": "mel-frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": t_res / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"tc": "f32 via split 16-bit pairs (fp16 pairs forward, bf16 pairs for gradients; 3 tcgen05 MMA passes per product, fp32 accumulate)",
                  "bf16x3": "as tc", "fp32": "f32"}[args.math], "data": "synthetic",
        "config": {"workload": WORKLOAD % args.preset + ", random-init weights, fwd+losses+bwd+clip+Adam",
                   "global_batch": B * world, "parallelism": "dp%d" % world,
                   "l2": "inputs larger than L2 (>1.5 GB touched per step)",
                   "cuda_graph": not args.no_graph, "conv_math": args.math,
                   "conv_math_note": {"tc": "tcgen05: forward operands as fp16 (hi, lo*2^11) pairs = 22-bit operands, "
                                            "gradient GEMMs on bf16 pairs (16 bits, full fp32 range), hi*hi + hi*lo + lo*hi "
                                            "with fp32 accumulation in TMEM; all three presets within rtol 1e-3 / atol 1e-4 of the "
                                            "fp32 oracle at B=16, full depth (tests/test_gpu_models.py)",
                                      "bf16x3": "alias of tc",
                                      "fp32": "exact fp32 FMA on CUDA cores"}[args.math]},
        "e2e": {"value": frames * args.steps / t_e2e, "unit": "mel-frames/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": t_e2e / args.steps * 1e3},
        "gpu_launches": int(launches), "loss": loss_val, "clocks": clocks.summary(),
    }
    del step, resident
    torch.cuda.empty_cache()

    # ---- the other two BASELINE presets (configs #3, #4), same step, every rank participates --------------------
    if not args.no_extras:
        presets = {}
        for name in [n for n in ("nyanko_ljspeech", "deepvoice3_vctk") if n != args.preset]:
            st, hb = make_step(name, args.math)
            rb = to_device(hb, dev)
            for _ in range(3):
                st.step(rb)
            t = timed(lambda: st.step(rb), 10)
            presets[name] = {"ms_per_step": t / 10 * 1e3, "value": frames * 10 / t, "unit": "mel-frames/s",
                             "n_gpus": world, "steps": 10}
            del st, rb
            torch.cuda.empty_cache()
        out["presets"] = presets
        out["stft"] = stft_throughput(dev, world, rank, timed)
    ops.conv_math = args.math

    if rank == 0:
        pk, pk_kind = peaks()
        if args.math in ("tc", "bf16x3"):
            out["roofline"] = convblock_roofline(dev, pk, pk_kind)
        if world == 1 and not args.no_extras:
            # strict mode, driver-timed beside the headline: exact-fp32 CUDA-core kernels, same step
            st, hb = make_step(args.preset, "fp32")
            rb = to_device(hb, dev)
            for _ in range(3):
                st.step(rb)
            t = timed(lambda: st.step(rb), 5)
            out["fp32_exact"] = {"ms_per_step": t / 5 * 1e3, "value": B * T_MEL * 5 / t, "unit": "mel-frames/s",
                                 "steps": 5, "note": "DV3_CONV_MATH=fp32: every contraction on exact-fp32 CUDA-core kernels"}
            del st, rb
            torch.cuda.empty_cache()
            ops.conv_math = args.math
            # the GPU competitor: the UNMODIFIED reference modules + train.py loop in PyTorch eager on this B200
            eager = {}
            for tf32 in (False, True):
                try:
                    r = reference_train_throughput(args.preset, dev, steps=8, warmup=3, tf32=tf32)
                except Exception as ex:                     # never let the competitor break the headline line
                    r, eager["error"] = None, "%s: %s" % (type(ex).__name__, ex)
                if r is not None:
                    eager["tf32_on" if tf32 else "tf32_off"] = {"value": r[0], "unit": "mel-frames/s",
                                                                "ms_per_step": r[1] * 1e3, "steps": r[2]}
            eager["what"] = ("reference package + reference train.py train() loop (oracle/_ref), PyTorch %s eager, cuDNN / "
                             "cuBLAS, dropout on, same batch shape; step time by host clock around synchronised steps"
                             % torch.__version__)
            out["gpu_eager_baseline"] = eager
        if world == 1 and not args.no_cpu_baseline:
            c = cpu_arm(args.preset, steps=3, warmup=1, budget_s=25.0)
            out["cpu_baseline"] = {"value": c["value"], "unit": "mel-frames/s", "cores": c["cores"], "kind": c["kind"],
                                   "cpu": cpu_model(),
                                   "sample": "%d full steps of the same workload after 1 warm-up (bounded to ~25 s), "
                                             "median; %.2f s/step on %d threads; %s" % (
                                                 c["n"], c["sec"], c["cores"],
                                                 "reference package + train.py loop (oracle/_ref)"
                                                 if c["kind"] == "reference" else "oracle port")}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_PARAMS = 8 << 20          # parameters sampled into params_sample.npy: 32 MB of float32


def dump_outputs(out_dir, loss, model):
    """What the last timed step hands its caller: the loss (loss.npy, float64) and the updated parameters -- the
    parameters in model.parameters() order, flattened, at a fixed seeded sample of DUMP_PARAMS positions in
    increasing order (params_sample.npy, float32)."""
    os.makedirs(out_dir, exist_ok=True)
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    n = flat.numel()
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:min(n, DUMP_PARAMS)].sort().values
    np.save(os.path.join(out_dir, "loss.npy"), np.float64(loss.double().item()))
    np.save(os.path.join(out_dir, "params_sample.npy"), flat[idx.to(flat.device)].float().cpu().numpy())


def stft_throughput(dev, world, rank, timed):
    """BASELINE.json config #5 (10k synthetic 10 s clips @22.05 kHz), sharded round-robin over the ranks with no
    collective: every rank processes ceil(10000 / world) clips as resident batches of 256 -> clips/s of the whole job,
    device-resident and end to end (pinned H2D of the waveforms, D2H of linear + mel)."""
    from deepvoice3_pytorch_b200 import audio
    n_samples, nb = 220500, 256
    per_rank = (10000 + world - 1) // world
    iters = (per_rank + nb - 1) // nb
    gen = torch.Generator().manual_seed(100 + rank)
    host = (0.1 * torch.randn(nb, n_samples, generator=gen)).clamp_(-1, 1).pin_memory()
    wav = host.to(dev)
    frames = audio.num_frames(n_samples)
    lin_h = torch.empty(nb, frames, 513).pin_memory()
    mel_h = torch.empty(nb, frames, 80).pin_memory()
    audio.stft_mel_batch(wav)
    t_dev = timed(lambda: audio.stft_mel_batch(wav), iters)

    def e2e():
        w = host.to(dev, non_blocking=True)
        lin, mel = audio.stft_mel_batch(w)
        lin_h.copy_(lin, non_blocking=True)
        mel_h.copy_(mel, non_blocking=True)
    e2e()
    t_e2e = timed(e2e, iters)
    clips = iters * nb * world
    bytes_clip = 4.0 * (n_samples + frames * 513 + frames * 80)
    pk, _ = peaks()
    return {"metric": "STFT->linear+mel clips/s (10 s clips @22.05 kHz, 10k-clip job sharded over ranks)",
            "clips": clips, "value": clips / t_dev, "unit": "clips/s", "n_gpus": world,
            "e2e": {"value": clips / t_e2e, "unit": "clips/s", "h2d_bytes_per_batch": int(host.numel() * 4),
                    "d2h_bytes_per_batch": int((lin_h.numel() + mel_h.numel()) * 4)},
            "hbm_gbs": bytes_clip * clips / world / t_dev / 1e9, "hbm_frac": bytes_clip * clips / world / t_dev / 1e9 / pk["hbm_gbs"],
            "parity": "unpinned (lws / librosa are un-vendored dependencies of the reference; oracle/audio_oracle.py)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", default="deepvoice3_ljspeech", choices=sorted(PRESETS))
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--math", default=os.environ.get("DV3_CONV_MATH", "tc"), choices=["tc", "fp32", "bf16x3"],
                    help="contraction arithmetic: tc = tcgen05 split 16-bit pairs (fp32-class, default), fp32 = CUDA cores")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the sub-benchmarks (other presets, STFT, exact-fp32 mode, reference-in-eager competitor)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and a fixed sample of the updated parameters of the "
                         "last timed step to DIR/*.npy (same arguments -> same inputs, for comparing two builds)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
