"""torch.autograd Functions over the dv3b200 C ABI (include/dv3b200.h).

PyTorch is plumbing here: it owns device memory, the current stream and autograd bookkeeping.  All
arithmetic happens in csrc/*.cu.  Every function requires CUDA fp32 tensors and raises otherwise --
there is no CPU fallback.
"""
import ctypes
import os

import torch

from ._lib import lib, Dv3Error

MODE_GLU, MODE_HIGHWAY = 0, 1

# Arithmetic of the ConvBlock / conv / attention contractions:
#   "tc"     (default) tcgen05 tensor cores, every fp32 operand split into a 16-bit (hi, lo) pair, hi*hi + hi*lo + lo*hi
#            with fp32 accumulation in TMEM (csrc/tc_gemm.cu, tc_attn.cu): fp16 pairs (22-bit operands) in the forward
#            GEMMs, bf16 pairs in the gradient GEMMs.  Full-depth preset models match the fp32 oracle at rtol 1e-3 /
#            atol 1e-4 (tests/test_gpu_models.py).  Shapes the tensor-core kernels do not cover (C % 128 != 0, tiny
#            GEMMs) run on the exact-fp32 kernels automatically.  ("bf16x3" is accepted as an alias.)
#   "fp32"   exact-fp32 CUDA-core kernels everywhere (csrc/conv.cu, bgemm.cu): ~7x slower, the strict reference mode.
conv_math = os.environ.get("DV3_CONV_MATH", "tc")


# ----------------------------------------------------------------------------------------------
# plumbing
# ----------------------------------------------------------------------------------------------
def _chk(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise Dv3Error("dv3b200 ops need CUDA tensors (got %s); there is no CPU path" % t.device)
        if t.dtype != torch.float32:
            raise Dv3Error("dv3b200 ops are fp32 (got %s)" % t.dtype)
        if not t.is_contiguous():
            raise Dv3Error("dv3b200 ops need contiguous tensors")


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


class DropoutState:
    """Step seed in device memory + call-site salts.

    keep(i) = f(seed[0], salt, i).  ``base`` is a persistent int64[1] device tensor that is bumped IN PLACE at the
    start of every training forward (a device-side add, so a captured CUDA graph gets fresh masks on every replay);
    ``seed`` is the snapshot of it that the kernels of the current forward -- and of its backward, through the
    autograd contexts, which hold the tensor -- read.  Salts are handed out in call order and restart with every
    outermost forward (``begin_forward``), so a replayed graph sees the same sequence."""

    GOLD = 0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF

    def __init__(self):
        self.base = None
        self.seed = None
        self.salt = 0
        self.depth = 0

    def _init(self, s, device):
        self.base = torch.tensor([int(s) & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device=device)
        self.seed = self.base.clone()

    def seed_tensor(self, device):
        if self.seed is None or self.seed.device != device:
            s = torch.initial_seed()
            if torch.distributed.is_available() and torch.distributed.is_initialized():
                s += 0x632BE59BD9B4E019 * torch.distributed.get_rank()      # different masks on every replica
            self._init(s, device)
        return self.seed

    def manual_seed(self, s, device):
        self._init(s, device)

    def next_salt(self):
        self.salt += 1
        return self.salt

    def start_forward(self):
        self.salt = 0

    def advance(self):
        """New masks from here on: bump the persistent seed in place, snapshot it for the coming forward."""
        if self.base is not None:
            self.base.add_(self.GOLD)
            self.seed = self.base.clone()

    # -- called by the model containers around their forward ------------------------------------------------
    def begin_forward(self, training, device):
        """Outermost forward of a model (or of model.seq2seq / model.postnet called on their own, reference
        train.py:691-700): restart the salts and, in training, draw a new step seed."""
        self.depth += 1
        if self.depth == 1:
            self.salt = 0
            if training and device.type == "cuda":
                self.seed_tensor(device)
                self.advance()

    def end_forward(self):
        self.depth -= 1


rng = DropoutState()


def forward_scope(fn):
    """Decorator for the ``forward`` of a module the reference's train.py may call on its own (model.postnet,
    train.py:700): draws the dropout seed / restarts the salts when it is the outermost forward."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, x, *a, **kw):
        rng.begin_forward(self.training, x.device)
        try:
            return fn(self, x, *a, **kw)
        finally:
            rng.end_forward()
    return wrapped


def _drop_args(p, training, device):
    """-> (p_eff, seed tensor | None, salt) ; consumes a salt only when dropout is live."""
    if training and p > 0.0:
        return float(p), rng.seed_tensor(device), rng.next_salt()
    return 0.0, None, 0


# ----------------------------------------------------------------------------------------------
# weight-norm packing helpers
# ----------------------------------------------------------------------------------------------
def _wn_conv_fwd(v, g):
    """v (Cout, Cin, k), g (Cout,1,1) -> w_f [k][Cin][Cout], w_b [k][Cout][Cin], inv_norm [Cout]."""
    Cout, Cin, k = v.shape
    w_f = torch.empty(k, Cin, Cout, device=v.device, dtype=torch.float32)
    w_b = torch.empty(k, Cout, Cin, device=v.device, dtype=torch.float32)
    inv = torch.empty(Cout, device=v.device, dtype=torch.float32)
    scale = torch.empty_like(inv)
    lib.call("dv3_weightnorm_fwd", _p(v), _p(g), _p(inv), _p(scale), _p(w_f), _p(w_b), Cout, Cin, k,
             1, Cout, Cin * Cout, Cin, 1, Cout * Cin, _stream())
    return w_f, w_b, inv


# Gradient sink (set by train_step.TrainStep): parameter gradients are accumulated by the kernels straight into the
# pre-allocated ``.grad`` views of the flat gradient arena and the autograd Functions return None for them, which
# removes one ``grad += new`` elementwise kernel per parameter per step (~130 launches).  Off by default: plain
# autograd semantics (Functions return dv, dg, dbias).
grad_sink = False


# Gradient-bucket boundaries (set by train_step.TrainStep in data-parallel runs): ``grad_boundary(x, tag)`` marks a tensor
# whose gradient, once computed, proves that every parameter gradient of the layers AFTER it is final -- the training
# step then starts the NCCL all-reduce of that parameter bucket while the rest of the backward pass still runs.
grad_boundary_cb = None


def grad_boundary(x, tag):
    if grad_boundary_cb is not None and x.requires_grad:
        cb = grad_boundary_cb

        def _hook(grad, tag=tag, cb=cb):
            cb(tag)
            return None
        x.register_hook(_hook)
    return x


# Batched weight norm (weight_bank.WeightBank), installed by train_step.TrainStep for the duration of one
# forward/backward: operand planes of every layer are prepared up front, the weight-norm backward is deferred to one
# launch after loss.backward().  None: every Function normalises / reduces its own layer.
weight_bank = None


def _bank_weights(v, g):
    return weight_bank.weights_for(v, g) if weight_bank is not None else None


def _sink(*params):
    """The .grad buffers to accumulate into, or None when the sink is off / not every buffer exists."""
    if not grad_sink or any(p.grad is None or not p.grad.is_contiguous() for p in params):
        return None
    return [p.grad for p in params]


def _wn_bwd(partials, nsplit, v, g, inv, tap_major_k=0, out=None, accumulate=False):
    """tap_major_k = 0: partials in v's layout; = k (> 0): partials as [j][R][X] (tensor-core weight gradient)."""
    dv, dg = out if out is not None else (torch.empty_like(v), torch.empty_like(g))
    R = v.shape[0]
    if tap_major_k:
        X = v.numel() // R // tap_major_k
        lib.call("dv3_weightnorm_bwd", _p(partials), v.numel(), nsplit, 1, _p(v), _p(g), _p(inv), _p(dv), _p(dg), R, X,
                 tap_major_k, int(accumulate), _stream())
    else:
        X = v.numel() // R
        lib.call("dv3_weightnorm_bwd", _p(partials), v.numel(), nsplit, 0, _p(v), _p(g), _p(inv), _p(dv), _p(dg), R, X,
                 1, int(accumulate), _stream())
    return dv, dg


def _wgrad_conv(dab, x, v_shape, k, dilation, causal, p, seed_ptr, salt):
    """partials [nsplit][Cout*Cin*k] in v's layout (Cout, Cin, k)."""
    B, M, T = dab.shape
    Cin = x.shape[1]
    nsplit = lib.raw("dv3_conv1d_wgrad_nsplit")(B, M, Cin, T, k)
    numel = M * Cin * k
    partials = torch.empty(nsplit, numel, device=x.device, dtype=torch.float32)
    lib.call("dv3_conv1d_wgrad", _p(dab), _p(x), _p(partials), numel, B, M, Cin, T, k, dilation,
             int(causal), p, seed_ptr, salt, M, Cin * k, 0, k, 1, _stream())
    return partials, nsplit


# ----------------------------------------------------------------------------------------------
# fused ConvBlock (Conv1dGLU / HighwayConv1d)
# ----------------------------------------------------------------------------------------------
class _ConvBlockFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, v, g, bias, spk, k, dilation, causal, mode, residual, p_drop, training):
        _chk(x, v, g, bias, spk)
        B, C, T = x.shape
        assert v.shape == (2 * C, C, k), "ConvBlock needs in_channels == out_channels"
        w_f, w_b, inv = _wn_conv_fwd(v, g)
        p, seed_t, salt = _drop_args(p_drop, training, x.device)
        seed_ptr = _p(seed_t)
        need_bwd = any(ctx.needs_input_grad)
        y = torch.empty_like(x)
        a = torch.empty_like(x) if need_bwd else None
        s = torch.empty_like(x) if need_bwd else None
        lib.call("dv3_convblock_fwd", _p(x), _p(w_f), _p(bias), _p(spk), _p(y), _p(a), _p(s), B, C, T, k,
                 dilation, int(causal), mode, int(residual), p, seed_ptr, salt, _stream())
        if need_bwd:
            ctx.save_for_backward(x, v, g, a, s, w_b, inv)
            ctx.cfg = (k, dilation, causal, mode, residual, p, salt, spk is not None, x.device)
            ctx.seed_t = seed_t
        return y

    @staticmethod
    def backward(ctx, dy):
        x, v, g, a, s, w_b, inv = ctx.saved_tensors
        k, dilation, causal, mode, residual, p, salt, has_spk, dev = ctx.cfg
        seed_ptr = _p(ctx.seed_t)          # the forward's own seed snapshot
        dy = _c(dy)
        B, C, T = x.shape
        dab = torch.empty(B, 2 * C, T, device=dev, dtype=torch.float32)
        dbias = torch.zeros(2 * C, device=dev, dtype=torch.float32)
        lib.call("dv3_convblock_gate_bwd", _p(dy), _p(a), _p(s), _p(x), _p(dab), _p(dbias), B, C, T, mode,
                 int(residual), _stream())
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            if mode == MODE_GLU:
                addmode, e1, e2, alpha = (1, dy, None, 0.7071067811865476) if residual else (0, None, None, 0.0)
            else:
                addmode, e1, e2, alpha = 2, dy, s, 0.0
            lib.call("dv3_conv1d_dgrad", _p(dab), _p(w_b), _p(dx), B, 2 * C, C, T, k, dilation,
                     int(causal), p, seed_ptr, salt, addmode, _p(e1), _p(e2), alpha, _stream())
        dv = dg = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            partials, nsplit = _wgrad_conv(dab, x, v.shape, k, dilation, causal, p, seed_ptr, salt)
            dv, dg = _wn_bwd(partials, nsplit, v, g, inv)
        dspk = dab[:, :C, :] if has_spk and ctx.needs_input_grad[4] else None
        return dx, dv, dg, dbias, dspk, None, None, None, None, None, None, None


# The weight-gradient GEMM (+ the weight-norm backward that consumes it) and the data-gradient GEMM of a block are
# independent: run the former on a side stream so the two overlap -- most layers launch only 32-128 CTAs on 148 SMs.
# Fork/join with stream waits, which a CUDA-graph capture records as graph edges.
overlap_wgrad = os.environ.get("DV3_OVERLAP_WGRAD", "1") == "1"
_side_streams = {}


class _SideStream:
    """with _SideStream(dev): ...   work inside is ordered after everything already on the current stream; the
    current stream waits for it at join()."""

    def __init__(self, dev):
        self.enabled = overlap_wgrad
        if self.enabled:
            if dev not in _side_streams:
                _side_streams[dev] = torch.cuda.Stream(device=dev)
            self.side = _side_streams[dev]
            self.main = torch.cuda.current_stream(dev)
            self.ctx = torch.cuda.stream(self.side)

    def __enter__(self):
        if self.enabled:
            self.side.wait_stream(self.main)
            self.ctx.__enter__()
        return self

    def __exit__(self, *a):
        if self.enabled:
            self.ctx.__exit__(*a)

    def join(self):
        if self.enabled:
            self.main.wait_stream(self.side)


def _pad8(n):
    return (n + 7) // 8 * 8


class _ConvBlockTCFn(torch.autograd.Function):
    """Same contract as _ConvBlockFn on the tcgen05 path: operands are bf16 hi/lo planes."""

    @staticmethod
    def forward(ctx, x, v, g, bias, spk, k, dilation, causal, mode, residual, p_drop, training):
        _chk(x, v, g, bias, spk)
        B, C, T = x.shape
        dev = x.device
        bf = torch.bfloat16
        need_bwd = any(ctx.needs_input_grad)
        bank = _bank_weights(v, g)        # operand planes already prepared for the whole model this step?
        if bank is not None:
            inv, wfwd, wbwd = bank.inv, bank.wfwd, bank.wbwd
        else:
            inv = torch.empty(2 * C, device=dev)
            scale = torch.empty_like(inv)
            wfwd = torch.empty(2, k, 2 * C, C, device=dev, dtype=torch.float16)
            wbwd = torch.empty(2, k, C, 2 * C, device=dev, dtype=bf)
        p, seed_t, salt = _drop_args(p_drop, training, dev)
        x_btc = torch.empty(2, B, T, C, device=dev, dtype=torch.float16)        # forward operand (fp16 pair)
        x_wg = torch.empty(2, B, T, C, device=dev, dtype=bf) if need_bwd else None  # weight-gradient operand
        seed_ptr = _p(seed_t)
        y = torch.empty_like(x)
        a = torch.empty_like(x) if need_bwd else None
        s = torch.empty_like(x) if need_bwd else None
        side = None
        if bank is None:
            side = _SideStream(dev)
            with side:                    # weight norm + split depends only on the parameters: overlap it with
                lib.call("dv3_tc_weightnorm_fwd", _p(v), _p(g), _p(inv), _p(scale), _p(wfwd), 2, _p(wbwd), 2 * C, C,
                         k, _stream())    # the activation split below
        lib.call("dv3_tc_split_input", _p(x), _p(x_btc), 2, _p(x_wg), B, C, T, k, dilation, int(causal), p,
                 seed_ptr, salt, _stream())
        if side is not None:
            side.join()
        lib.call("dv3_tc_convblock_fwd", _p(x_btc), _p(wfwd), 2, _p(bias), _p(spk), _p(x), _p(y), _p(a), _p(s),
                 B, C, T, k, dilation, int(causal), mode, int(residual), None, _stream())
        if need_bwd:
            ctx.save_for_backward(x, v, g, a, s, x_wg, wbwd, inv)
            ctx.cfg = (k, dilation, causal, mode, residual, p, salt, spk is not None, dev)
            ctx.seed_t = seed_t
            ctx.bias_param = bias if bias.is_leaf else None
            ctx.bank = bank
        return y

    @staticmethod
    def backward(ctx, dy):
        x, v, g, a, s, x_wg, wbwd, inv = ctx.saved_tensors
        k, dilation, causal, mode, residual, p, salt, has_spk, dev = ctx.cfg
        seed_ptr = _p(ctx.seed_t)          # the forward's own seed snapshot
        dy = _c(dy)
        B, C, T = x.shape
        bf = torch.bfloat16
        sink = _sink(v, g, ctx.bias_param) if ctx.bias_param is not None else None
        d_btc = torch.empty(2, B, T, 2 * C, device=dev, dtype=bf)
        dbias = sink[2] if sink else torch.zeros(2 * C, device=dev)
        lib.call("dv3_tc_gate_bwd_split", _p(dy), _p(a), _p(s), _p(x), _p(d_btc), None, _p(dbias), B, C, T,
                 mode, int(residual), _stream())
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        dv = dg = partials = None
        if need_w:                                   # allocate on the main stream, compute on the side stream
            nsplit = lib.raw("dv3_tc_wgrad_nsplit")(B, 2 * C, C, T, k)
            numel = v.numel()
            # with the weight bank the split-K partials go to the layer's persistent buffer and the weight-norm
            # backward of ALL layers runs as one launch after loss.backward() (WeightBank.end_backward)
            partials = weight_bank.partials_for(ctx.bank, nsplit, numel) if (sink and ctx.bank is not None) else None
            deferred = partials is not None
            if not deferred:
                partials = torch.empty(nsplit, numel, device=dev)
            dv, dg = (sink[0], sink[1]) if sink else (torch.empty_like(v), torch.empty_like(g))
        side = _SideStream(dev)
        if need_w:
            with side:
                # partials [split][j][2C][C]: contiguous float4 stores from the GEMM epilogue
                lib.call("dv3_tc_wgrad_mn", _p(d_btc), _p(x_wg), _p(partials), numel, B, 2 * C, C, T, k, dilation,
                         int(causal), 2 * C, C, 0, 1, 2 * C * C, _stream())
                if not deferred:
                    _wn_bwd(partials, nsplit, v, g, inv, tap_major_k=k, out=(dv, dg), accumulate=bool(sink))
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            if mode == MODE_GLU:
                addmode, e1, e2, alpha = (1, dy, None, 0.7071067811865476) if residual else (0, None, None, 0.0)
            else:
                addmode, e1, e2, alpha = 2, dy, s, 0.0
            lib.call("dv3_tc_conv", _p(d_btc), _p(wbwd), 2, _p(dx), B, 2 * C, C, T, k, dilation, int(causal), 1,
                     None, 0, p, seed_ptr, salt, addmode, _p(e1), _p(e2), alpha, None, _stream())
        if need_w:
            side.join()
        if sink:                                     # already accumulated into the .grad arena views
            dv = dg = dbias = None
        dspk = None
        if has_spk and ctx.needs_input_grad[4]:     # d_a = hi + lo * 2^-11 of the (B,T,2C) planes, back to (B,C,T)
            dspk = transpose12((d_btc[0, :, :, :C].float() + d_btc[1, :, :, :C].float() * (1.0 / 2048.0)).contiguous())
        return (dx, dv, dg, dbias, dspk) + (None,) * 7


class _Conv1dTCFn(torch.autograd.Function):
    """Plain weight-normed conv (+ReLU) on the tcgen05 path (1x1 convs, projections)."""

    @staticmethod
    def forward(ctx, x, v, g, bias, k, dilation, causal, relu):
        _chk(x, v, g, bias)
        B, Cin, T = x.shape
        Cout = v.shape[0]
        dev, bf = x.device, torch.bfloat16
        need_bwd = any(ctx.needs_input_grad)
        Cinp, Coutp = _pad8(Cin), _pad8(Cout)
        bank = _bank_weights(v, g)
        if bank is not None:
            inv, wfwd, wbwd = bank.inv, bank.wfwd, bank.wbwd
        else:
            inv = torch.empty(Cout, device=dev)
            scale = torch.empty_like(inv)
            wfwd = torch.empty(2, k, Cout, Cinp, device=dev, dtype=torch.float16)
            wbwd = torch.empty(2, k, Cin, Coutp, device=dev, dtype=bf)
        need_w = need_bwd and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        x_btc = torch.empty(2, B, T, Cinp, device=dev, dtype=torch.float16)
        x_wg = torch.empty(2, B, T, Cinp, device=dev, dtype=bf) if need_w else None
        y = torch.empty(B, Cout, T, device=dev)
        side = None
        if bank is None:
            side = _SideStream(dev)
            with side:
                lib.call("dv3_tc_weightnorm_fwd", _p(v), _p(g), _p(inv), _p(scale), _p(wfwd), 2, _p(wbwd), Cout, Cin,
                         k, _stream())
        lib.call("dv3_tc_split_input", _p(x), _p(x_btc), 2, _p(x_wg), B, Cin, T, k, dilation, int(causal), 0.0,
                 None, 0, _stream())
        if side is not None:
            side.join()
        lib.call("dv3_tc_conv", _p(x_btc), _p(wfwd), 2, _p(y), B, Cin, Cout, T, k, dilation, int(causal), 0,
                 _p(bias), int(relu), 0.0, None, 0, 0, None, None, 0.0, None, _stream())
        if need_bwd:
            ctx.save_for_backward(v, g, x_wg, wbwd, inv, y if relu else None)
            ctx.cfg = (B, Cin, Cout, T, k, dilation, causal, relu)
            ctx.bias_param = bias if bias.is_leaf else None
            ctx.bank = bank
        return y

    @staticmethod
    def backward(ctx, dy):
        v, g, x_wg, wbwd, inv, y = ctx.saved_tensors
        B, Cin, Cout, T, k, dilation, causal, relu = ctx.cfg
        dy = _c(dy)
        dev, bf = dy.device, torch.bfloat16
        Coutp = _pad8(Cout)
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        sink = _sink(v, g, ctx.bias_param) if (ctx.bias_param is not None and v.is_leaf and g.is_leaf) else None
        g_btc = torch.empty(2, B, T, Coutp, device=dev, dtype=bf)
        dbias = sink[2] if sink else torch.zeros(Cout, device=dev)
        lib.call("dv3_tc_grad_split", _p(dy), _p(y), _p(g_btc), None, _p(dbias), B, Cout, T, int(relu), _stream())
        dv = dg = None
        side = _SideStream(dev)
        if need_w:
            nsplit = lib.raw("dv3_tc_wgrad_nsplit")(B, Cout, Cin, T, k)
            numel = v.numel()
            partials = weight_bank.partials_for(ctx.bank, nsplit, numel) if (sink and ctx.bank is not None) else None
            deferred = partials is not None
            if not deferred:
                partials = torch.empty(nsplit, numel, device=dev)
            dv, dg = (sink[0], sink[1]) if sink else (torch.empty_like(v), torch.empty_like(g))
            with side:
                lib.call("dv3_tc_wgrad_mn", _p(g_btc), _p(x_wg), _p(partials), numel, B, Cout, Cin, T, k, dilation,
                         int(causal), Cout, Cin, 0, 1, Cout * Cin, _stream())
                if not deferred:
                    _wn_bwd(partials, nsplit, v, g, inv, tap_major_k=k, out=(dv, dg), accumulate=bool(sink))
        dx = None
        if need_x:
            dx = torch.empty(B, Cin, T, device=dev)
            lib.call("dv3_tc_conv", _p(g_btc), _p(wbwd), 2, _p(dx), B, Cout, Cin, T, k, dilation, int(causal), 1, None,
                     0, 0.0, None, 0, 0, None, None, 0.0, None, _stream())
        if need_w:
            side.join()
        if sink:
            dv = dg = dbias = None
        return (dx, dv, dg, dbias) + (None,) * 4


class _ConvT2TCFn(torch.autograd.Function):
    """ConvTranspose1d(k=2,s=2) on the tcgen05 path: a 1x1 conv with 2*Cout rows (j,co) + the time interleave."""

    @staticmethod
    def forward(ctx, x, v, g, bias):
        _chk(x, v, g, bias)
        B, Cin, T = x.shape
        Cout = v.shape[1]
        dev, bf = x.device, torch.bfloat16
        Cinp, K2p = _pad8(Cin), _pad8(2 * Cout)
        inv = torch.empty(Cin, device=dev)
        scale = torch.empty_like(inv)
        wfwd = torch.empty(2, 2 * Cout, Cinp, device=dev, dtype=torch.float16)
        wbwd = torch.empty(2, Cin, K2p, device=dev, dtype=bf)
        lib.call("dv3_tc_weightnorm_convt_fwd", _p(v), _p(g), _p(inv), _p(scale), _p(wfwd), 2, _p(wbwd), Cin, Cout,
                 _stream())
        x_btc = torch.empty(2, B, T, Cinp, device=dev, dtype=torch.float16)
        x_wg = torch.empty(2, B, T, Cinp, device=dev, dtype=bf)
        lib.call("dv3_tc_split_input", _p(x), _p(x_btc), 2, _p(x_wg), B, Cin, T, 1, 1, 0, 0.0, None, 0, _stream())
        bias2 = bias.repeat(2)
        yp = torch.empty(B, 2 * Cout, T, device=dev)
        lib.call("dv3_tc_conv", _p(x_btc), _p(wfwd), 2, _p(yp), B, Cin, 2 * Cout, T, 1, 1, 0, 0, _p(bias2), 0, 0.0,
                 None, 0, 0, None, None, 0.0, None, _stream())
        y = torch.empty(B, Cout, 2 * T, device=dev)
        lib.call("dv3_interleave2", _p(yp), _p(y), B, Cout, T, 0, _stream())
        ctx.save_for_backward(v, g, x_wg, wbwd, inv)
        ctx.cfg = (B, Cin, Cout, T)
        return y

    @staticmethod
    def backward(ctx, dy):
        v, g, x_wg, wbwd, inv = ctx.saved_tensors
        B, Cin, Cout, T = ctx.cfg
        dy = _c(dy)
        dev, bf = dy.device, torch.bfloat16
        K2p = _pad8(2 * Cout)
        dyp = torch.empty(B, 2 * Cout, T, device=dev)
        lib.call("dv3_interleave2", _p(dy), _p(dyp), B, Cout, T, 1, _stream())
        g_btc = torch.empty(2, B, T, K2p, device=dev, dtype=bf)
        db2 = torch.zeros(2 * Cout, device=dev)
        lib.call("dv3_tc_grad_split", _p(dyp), None, _p(g_btc), None, _p(db2), B, 2 * Cout, T, 0, _stream())
        dbias = db2[:Cout] + db2[Cout:]
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(B, Cin, T, device=dev)
            lib.call("dv3_tc_conv", _p(g_btc), _p(wbwd), 2, _p(dx), B, 2 * Cout, Cin, T, 1, 1, 0, 1, None, 0, 0.0, None,
                     0, 0, None, None, 0.0, None, _stream())
        dv = dg = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            M = 2 * Cout
            nsplit = lib.raw("dv3_tc_wgrad_nsplit")(B, M, Cin, T, 1)
            numel = v.numel()
            partials = torch.empty(nsplit, numel, device=dev)
            # element (m=(j,co), ci) -> v layout (ci, co, j): ci*2*Cout + co*2 + j
            lib.call("dv3_tc_wgrad_mn", _p(g_btc), _p(x_wg), _p(partials), numel, B, M, Cin, T, 1, 1, 0, Cout, 2, 1,
                     2 * Cout, 0, _stream())
            dv, dg = _wn_bwd(partials, nsplit, v, g, inv)
        return dx, dv, dg, dbias


# 16 keeps the 16-wide speaker projections of the multi-speaker model on tensor cores (measured: vctk step 11.8 -> 10.6 ms)
TC_MIN_CHANNELS = int(os.environ.get("DV3_TC_MIN_CHANNELS", "16"))


def _use_tc_conv(x, Cin, Cout, k):
    """Tensor cores for plain convs when the mode asks for it, the shape is supported and the GEMM is big enough to
    amortise the operand-split passes."""
    if conv_math not in ("tc", "bf16x3") or not x.is_cuda:
        return False
    B, _, T = x.shape
    if not lib.raw("dv3_tc_conv_supported")(B, Cin, Cout, T, int(k)):
        return False
    if k > 1 and Cin % 128 != 0:          # the data gradient swaps the roles of Cin / Cout
        return False
    return min(Cin, Cout) >= TC_MIN_CHANNELS and B * T >= 512


def tc_supported(B, C, T, k):
    return bool(lib.raw("dv3_tc_supported")(B, C, T, k))


def convblock(x, v, g, bias, spk=None, k=3, dilation=1, causal=False, mode=MODE_GLU, residual=True,
              p_drop=0.0, training=False):
    """Fused weight-normed dilated conv + gate.  x (B,C,T); v (2C,C,k); g (2C,1,1); bias (2C);
    spk (B,C,T) already softsign'ed (or None)."""
    if conv_math in ("tc", "bf16x3") and x.is_cuda and tc_supported(x.shape[0], x.shape[1], x.shape[2], int(k)):
        return _ConvBlockTCFn.apply(_c(x), v, g, bias, None if spk is None else _c(spk), int(k), int(dilation),
                                    bool(causal), int(mode), bool(residual), float(p_drop), bool(training))
    if conv_math not in ("fp32", "bf16x3", "tc"):
        raise Dv3Error("unknown conv_math %r" % (conv_math,))
    return _ConvBlockFn.apply(_c(x), v, g, bias, None if spk is None else _c(spk), int(k), int(dilation),
                              bool(causal), int(mode), bool(residual), float(p_drop), bool(training))


# ----------------------------------------------------------------------------------------------
# plain weight-normed Conv1d (+ReLU)
# ----------------------------------------------------------------------------------------------
class _Conv1dFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, v, g, bias, k, dilation, causal, relu):
        _chk(x, v, g, bias)
        B, Cin, T = x.shape
        Cout = v.shape[0]
        assert v.shape == (Cout, Cin, k)
        w_f, w_b, inv = _wn_conv_fwd(v, g)
        y = torch.empty(B, Cout, T, device=x.device, dtype=torch.float32)
        lib.call("dv3_conv1d_fwd", _p(x), _p(w_f), _p(bias), _p(y), B, Cin, Cout, T, k, dilation,
                 int(causal), int(relu), _stream())
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(x, v, g, w_b, inv, y if relu else None)
            ctx.cfg = (k, dilation, causal, relu)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, v, g, w_b, inv, y = ctx.saved_tensors
        k, dilation, causal, relu = ctx.cfg
        dy = _c(dy)
        B, Cin, T = x.shape
        Cout = v.shape[0]
        dbias = torch.zeros(Cout, device=x.device, dtype=torch.float32)
        dyr = torch.empty_like(dy) if relu else dy
        lib.call("dv3_bias_act_bwd", _p(dy), _p(y), _p(dyr), _p(dbias), B, Cout, T, int(relu), _stream())
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            lib.call("dv3_conv1d_dgrad", _p(dyr), _p(w_b), _p(dx), B, Cout, Cin, T, k, dilation, int(causal),
                     0.0, None, 0, 0, None, None, 0.0, _stream())
        dv = dg = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            partials, nsplit = _wgrad_conv(dyr, x, v.shape, k, dilation, causal, 0.0, None, 0)
            dv, dg = _wn_bwd(partials, nsplit, v, g, inv)
        return dx, dv, dg, dbias, None, None, None, None


def conv1d(x, v, g, bias, k=1, dilation=1, causal=False, relu=False):
    """Weight-normed Conv1d with 'same' (or causal) padding, optional fused ReLU.  x (B,Cin,T)."""
    if _use_tc_conv(x, v.shape[1], v.shape[0], k):
        return _Conv1dTCFn.apply(_c(x), v, g, bias, int(k), int(dilation), bool(causal), bool(relu))
    return _Conv1dFn.apply(_c(x), v, g, bias, int(k), int(dilation), bool(causal), bool(relu))


# ----------------------------------------------------------------------------------------------
# layout, lookups, position encodings, dropout
# ----------------------------------------------------------------------------------------------
class _TransposeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _chk(x)
        B, R, C = x.shape
        y = torch.empty(B, C, R, device=x.device, dtype=torch.float32)
        lib.call("dv3_transpose", _p(x), _p(y), B, R, C, _stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = _c(dy)
        B, C, R = dy.shape
        dx = torch.empty(B, R, C, device=dy.device, dtype=torch.float32)
        lib.call("dv3_transpose", _p(dy), _p(dx), B, C, R, _stream())
        return dx


def transpose12(x):
    """(B, R, C) -> contiguous (B, C, R) -- the (B,T,C) <-> (B,C,T) layout change."""
    return _TransposeFn.apply(_c(x))


_err_flags = {}


def _err_flag(device):
    f = _err_flags.get(device)
    if f is None:
        f = torch.zeros(1, dtype=torch.int32, device=device)
        _err_flags[device] = f
    return f


def check_index_errors(device=None):
    """Raise if any lookup kernel saw an out-of-range id since the last call (one D2H sync)."""
    for dev, f in _err_flags.items():
        if device is not None and dev != device:
            continue
        if int(f.item()) != 0:
            f.zero_()
            raise IndexError("dv3b200: embedding / position index out of range")


class _EmbeddingFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ids, table, padding_idx):
        _chk(table)
        assert ids.dtype == torch.int64 and ids.is_cuda
        ids = ids.contiguous()
        N, (V, D) = ids.numel(), table.shape
        out = torch.empty(*ids.shape, D, device=table.device, dtype=torch.float32)
        lib.call("dv3_embedding_fwd", _p(ids), _p(table), _p(out), N, D, V, _p(_err_flag(table.device)),
                 _stream())
        ctx.save_for_backward(ids)
        ctx.cfg = (V, D, -1 if padding_idx is None else int(padding_idx))
        return out

    @staticmethod
    def backward(ctx, dy):
        (ids,) = ctx.saved_tensors
        V, D, pad = ctx.cfg
        dy = _c(dy)
        dtable = torch.zeros(V, D, device=dy.device, dtype=torch.float32)
        lib.call("dv3_embedding_bwd", _p(ids), _p(dy), _p(dtable), ids.numel(), D, V, pad, _stream())
        return None, dtable, None


def embedding(ids, table, padding_idx=None):
    return _EmbeddingFn.apply(ids, table, padding_idx)


class _SinusoidFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, table, w):
        _chk(table, w)
        assert pos.dtype == torch.int64 and pos.is_cuda and pos.dim() == 2
        pos = pos.contiguous()
        B, T = pos.shape
        P, D = table.shape
        out = torch.empty(B, T, D, device=table.device, dtype=torch.float32)
        lib.call("dv3_sinusoid_fwd", _p(pos), _p(table), _p(w), w.numel(), _p(out), B, T, D, P,
                 _p(_err_flag(table.device)), _stream())
        ctx.save_for_backward(pos, table, w)
        return out

    @staticmethod
    def backward(ctx, dy):
        pos, table, w = ctx.saved_tensors
        dy = _c(dy)
        B, T = pos.shape
        P, D = table.shape
        dtable = torch.zeros_like(table) if ctx.needs_input_grad[1] else None
        dw = torch.zeros_like(w) if ctx.needs_input_grad[2] else None
        if dtable is not None or dw is not None:
            lib.call("dv3_sinusoid_bwd", _p(pos), _p(table), _p(w), w.numel(), _p(dy), _p(dtable), _p(dw), B, T,
                     D, P, _stream())
        return None, dtable, dw


def sinusoidal_encoding(pos, table, w):
    """pos int64 (B,T); table (P,D) raw position table; w fp32 tensor with 1 or B position rates."""
    return _SinusoidFn.apply(pos, table, w)


class _DropoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p, seed_t, salt):
        _chk(x)
        y = torch.empty_like(x)
        lib.call("dv3_dropout", _p(x), _p(y), x.numel(), p, _p(seed_t), salt, _stream())
        ctx.cfg = (p, seed_t, salt)
        return y

    @staticmethod
    def backward(ctx, dy):
        p, seed_t, salt = ctx.cfg
        dy = _c(dy)
        dx = torch.empty_like(dy)
        lib.call("dv3_dropout", _p(dy), _p(dx), dy.numel(), p, _p(seed_t), salt, _stream())
        return dx, None, None, None


def dropout(x, p, training):
    if not training or p <= 0.0:
        return x
    return _DropoutFn.apply(_c(x), float(p), rng.seed_tensor(x.device), rng.next_salt())


# ----------------------------------------------------------------------------------------------
# ConvTranspose1d(k=2, stride=2) and Linear on the conv kernels
# ----------------------------------------------------------------------------------------------
class _ConvT2Fn(torch.autograd.Function):
    """y[b,co,2t+j] = bias[co] + sum_ci x[b,ci,t] w[ci,co,j]; w = g*v/||v|| over dim 0 (= Cin).
    Runs as a 1x1 conv with 2*Cout output rows ordered (j,co) followed by a time interleave."""

    @staticmethod
    def forward(ctx, x, v, g, bias):
        _chk(x, v, g, bias)
        B, Cin, T = x.shape
        Cout = v.shape[1]
        assert v.shape == (Cin, Cout, 2)
        dev = x.device
        w_f = torch.empty(Cin, 2 * Cout, device=dev, dtype=torch.float32)     # [ci][(j,co)]
        w_b = torch.empty(2 * Cout, Cin, device=dev, dtype=torch.float32)     # [(j,co)][ci]
        inv = torch.empty(Cin, device=dev, dtype=torch.float32)
        scale = torch.empty_like(inv)
        lib.call("dv3_weightnorm_fwd", _p(v), _p(g), _p(inv), _p(scale), _p(w_f), _p(w_b), Cin, Cout, 2,
                 2 * Cout, 1, Cout, 1, Cin, Cout * Cin, _stream())
        bias2 = bias.repeat(2)
        yp = torch.empty(B, 2 * Cout, T, device=dev, dtype=torch.float32)
        lib.call("dv3_conv1d_fwd", _p(x), _p(w_f), _p(bias2), _p(yp), B, Cin, 2 * Cout, T, 1, 1, 0, 0, _stream())
        y = torch.empty(B, Cout, 2 * T, device=dev, dtype=torch.float32)
        lib.call("dv3_interleave2", _p(yp), _p(y), B, Cout, T, 0, _stream())
        ctx.save_for_backward(x, v, g, w_b, inv)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, v, g, w_b, inv = ctx.saved_tensors
        dy = _c(dy)
        B, Cin, T = x.shape
        Cout = v.shape[1]
        dev = x.device
        dyp = torch.empty(B, 2 * Cout, T, device=dev, dtype=torch.float32)
        lib.call("dv3_interleave2", _p(dy), _p(dyp), B, Cout, T, 1, _stream())
        db2 = torch.zeros(2 * Cout, device=dev, dtype=torch.float32)
        lib.call("dv3_bias_act_bwd", _p(dyp), None, None, _p(db2), B, 2 * Cout, T, 0, _stream())
        dbias = db2[:Cout] + db2[Cout:]
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            lib.call("dv3_conv1d_dgrad", _p(dyp), _p(w_b), _p(dx), B, 2 * Cout, Cin, T, 1, 1, 0, 0.0, None, 0, 0,
                     None, None, 0.0, _stream())
        dv = dg = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            M = 2 * Cout
            nsplit = lib.raw("dv3_conv1d_wgrad_nsplit")(B, M, Cin, T, 1)
            numel = v.numel()
            partials = torch.empty(nsplit, numel, device=dev, dtype=torch.float32)
            # element (m=(j,co), ci) -> v layout (ci, co, j): co*2 + j + ci*Cout*2
            lib.call("dv3_conv1d_wgrad", _p(dyp), _p(x), _p(partials), numel, B, M, Cin, T, 1, 1, 0, 0.0, None, 0,
                     Cout, 2, 1, Cout * 2, 0, _stream())
            dv, dg = _wn_bwd(partials, nsplit, v, g, inv)
        return dx, dv, dg, dbias


def conv_transpose1d_k2s2(x, v, g, bias):
    if _use_tc_conv(x, v.shape[0], 2 * v.shape[1], 1):
        return _ConvT2TCFn.apply(_c(x), v, g, bias)
    return _ConvT2Fn.apply(_c(x), v, g, bias)


def linear(x, v, g, bias):
    """Weight-normed Linear over the last dim (reference modules.py:80-85): x (..., Cin) -> (..., Cout).
    Runs on the conv kernels in channel-major layout: (N,Cin) -> (1,Cin,N) -> 1x1 conv -> back."""
    shp = x.shape
    Cin, Cout = shp[-1], v.shape[0]
    x2 = x.reshape(1, -1, Cin)
    y = conv1d(transpose12(x2), v.view(Cout, Cin, 1), g.view(Cout, 1, 1), bias)
    return transpose12(y).reshape(*shp[:-1], Cout)


# ----------------------------------------------------------------------------------------------
# attention core (channel-major): q (B,E,Td), k (B,E,Ts), v (B,E,Ts) -> out (B,E,Td), probs (B,Td,Ts)
# ----------------------------------------------------------------------------------------------
def _bgemm(A, sA, Bm, sB, C, sCb, ldc, batch, M, N, K, alpha=1.0, accumulate=False):
    lib.call("dv3_bgemm", _p(A), sA[0], sA[1], sA[2], _p(Bm), sB[0], sB[1], sB[2], _p(C), sCb, ldc, batch, M, N,
             K, float(alpha), int(accumulate), _stream())


class _AttentionCoreFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, mask, p_drop, training):
        _chk(q, k, v)
        B, E, Td = q.shape
        Ts = k.shape[2]
        dev = q.device
        scores = torch.empty(B, Td, Ts, device=dev, dtype=torch.float32)
        # S[t,s] = sum_e q[e,t] k[e,s]                       (reference deepvoice3.py:143, no 1/sqrt(d))
        _bgemm(q, (E * Td, 1, Td), k, (E * Ts, Ts, 1), scores, Td * Ts, Ts, B, Td, Ts, E)
        p, seed_t, salt = _drop_args(p_drop, training, dev)
        seed_ptr = _p(seed_t)
        probs = torch.empty_like(scores)
        pd = torch.empty_like(scores) if p > 0 else None
        lib.call("dv3_softmax_fwd", _p(scores), _p(mask), _p(probs), _p(pd), B * Td, Ts, Td, p, seed_ptr, salt,
                 _stream())
        pv = pd if pd is not None else probs
        scale = Ts * (1.0 / Ts) ** 0.5                         # deepvoice3.py:170-171
        out = torch.empty(B, E, Td, device=dev, dtype=torch.float32)
        # O[e,t] = scale * sum_s v[e,s] pd[t,s]
        _bgemm(v, (E * Ts, Ts, 1), pv, (Td * Ts, 1, Ts), out, E * Td, Td, B, E, Td, Ts, alpha=scale)
        ctx.save_for_backward(q, k, v, probs, pd)
        ctx.cfg = (p, salt, scale)
        ctx.seed_t = seed_t
        ctx.mark_non_differentiable()
        return out, probs

    @staticmethod
    def backward(ctx, dout, dprobs_ext):
        q, k, v, probs, pd = ctx.saved_tensors
        p, salt, scale = ctx.cfg
        B, E, Td = q.shape
        Ts = k.shape[2]
        dev = q.device
        dout = _c(dout)
        seed_ptr = _p(ctx.seed_t)          # the forward's own seed snapshot
        pv = pd if pd is not None else probs
        # dPd[t,s] = scale * sum_e dO[e,t] v[e,s]
        dpd = torch.empty(B, Td, Ts, device=dev, dtype=torch.float32)
        _bgemm(dout, (E * Td, 1, Td), v, (E * Ts, Ts, 1), dpd, Td * Ts, Ts, B, Td, Ts, E, alpha=scale)
        # dV[e,s] = scale * sum_t dO[e,t] pd[t,s]
        dv = torch.empty_like(v)
        _bgemm(dout, (E * Td, Td, 1), pv, (Td * Ts, Ts, 1), dv, E * Ts, Ts, B, E, Ts, Td, alpha=scale)
        ds = torch.empty_like(dpd)
        dpe = _c(dprobs_ext) if dprobs_ext is not None else None
        lib.call("dv3_softmax_bwd", _p(probs), _p(dpd), _p(dpe), _p(ds), B * Td, Ts, p, seed_ptr, salt, _stream())
        # dq[e,t] = sum_s k[e,s] dS[t,s] ; dk[e,s] = sum_t q[e,t] dS[t,s]
        dq = torch.empty_like(q)
        _bgemm(k, (E * Ts, Ts, 1), ds, (Td * Ts, 1, Ts), dq, E * Td, Td, B, E, Td, Ts)
        dk = torch.empty_like(k)
        _bgemm(q, (E * Td, Td, 1), ds, (Td * Ts, Ts, 1), dk, E * Ts, Ts, B, E, Ts, Td)
        return dq, dk, dv, None, None, None


tc_attention = os.environ.get("DV3_TC_ATTN", "1") == "1"      # 0: attention on the exact-fp32 bgemm + softmax kernels


class _AttentionTCFn(torch.autograd.Function):
    """The same contract on the fused tcgen05 kernels (csrc/tc_attn.cu): one launch forward, two backward."""

    @staticmethod
    def forward(ctx, q, k, v, mask, p_drop, training):
        _chk(q, k, v)
        B, E, Td = q.shape
        Ts = k.shape[2]
        dev = q.device
        p, seed_t, salt = _drop_args(p_drop, training, dev)
        scale = Ts * (1.0 / Ts) ** 0.5                         # deepvoice3.py:170-171
        probs = torch.empty(B, Td, Ts, device=dev, dtype=torch.float32)
        out = torch.empty(B, E, Td, device=dev, dtype=torch.float32)
        lib.call("dv3_tc_attn_fwd", _p(q), _p(k), _p(v), _p(mask), _p(probs), _p(out), B, E, Td, Ts, scale, p,
                 _p(seed_t), salt, _stream())
        ctx.save_for_backward(q, k, v, probs)
        ctx.cfg = (p, salt, scale)
        ctx.seed_t = seed_t
        return out, probs

    @staticmethod
    def backward(ctx, dout, dprobs_ext):
        q, k, v, probs = ctx.saved_tensors
        p, salt, scale = ctx.cfg
        B, E, Td = q.shape
        Ts = k.shape[2]
        dev = q.device
        dout = _c(dout)
        dpe = _c(dprobs_ext) if dprobs_ext is not None else None
        ds = torch.empty(B, Td, Ts, device=dev, dtype=torch.float32)
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        lib.call("dv3_tc_attn_bwd", _p(dout), _p(q), _p(k), _p(v), _p(probs), _p(dpe), _p(ds), _p(dq), _p(dk), _p(dv),
                 B, E, Td, Ts, scale, p, _p(ctx.seed_t), salt, _stream())
        return dq, dk, dv, None, None, None


def attention_core(q, k, v, mask=None, p_drop=0.0, training=False):
    """mask: (B, Ts) uint8/bool, 1 = padding.  Returns (out (B,E,Td), probs (B,Td,Ts))."""
    if mask is not None:
        mask = mask.to(torch.uint8).contiguous()
    B, E, Td = q.shape
    tc = (conv_math in ("tc", "bf16x3") and tc_attention and q.is_cuda and
          lib.raw("dv3_tc_attn_supported")(B, E, Td, k.shape[2]))
    fn = _AttentionTCFn if tc else _AttentionCoreFn
    return fn.apply(_c(q), _c(k), _c(v), mask, float(p_drop), bool(training))
