"""Building blocks with the reference's names and call signatures (reference deepvoice3_pytorch/modules.py),
executing on the dv3b200 CUDA kernels.

Initialisation follows the reference factories draw-for-draw (a scratch torch module consumes the RNG the
way ``nn.Conv1d`` / ``nn.Linear`` would before ``normal_``), so ``torch.manual_seed(s)`` gives the same
initial model as the reference builder.
"""
import math

import numpy as np
import torch
from torch import nn
from torch.nn import functional as F

from . import ops
from .conv import Conv1d as _Conv1d, ConvTranspose1d as _ConvTranspose1d, WNLinear


def position_encoding_init(n_position, d_pos_vec, position_rate=1.0, sinusoidal=True):
    """Position table (reference modules.py:10-24): float64 arithmetic, cast to float32, then sin/cos
    on even/odd columns of rows >= 1 in float32.  Row 0 (padding position) stays zero."""
    pos = np.arange(n_position, dtype=np.float64).reshape(-1, 1)
    denom = np.power(10000, 2 * (np.arange(d_pos_vec) // 2) / d_pos_vec)
    enc = position_rate * pos / denom
    enc[0, :] = 0.0
    enc = torch.from_numpy(enc).float()
    if sinusoidal:
        enc[1:, 0::2] = torch.sin(enc[1:, 0::2])
        enc[1:, 1::2] = torch.cos(enc[1:, 1::2])
    return enc


class SinusoidalEncoding(nn.Embedding):
    """reference modules.py:34-64.  weight = raw (non-sinusoidal) table; forward(x, w) scales it by the
    position rate w (python scalar, or a (B,) tensor of per-utterance rates) and applies sin/cos."""

    def __init__(self, num_embeddings, embedding_dim, *args, **kwargs):
        super().__init__(num_embeddings, embedding_dim, padding_idx=0, *args, **kwargs)
        self.weight.data = position_encoding_init(num_embeddings, embedding_dim, position_rate=1.0,
                                                  sinusoidal=False)

    def _rate_tensor(self, w):
        """Scalar rates are cached as 1-element device tensors (no H2D copy per call: graph-capture safe)."""
        cache = self.__dict__.setdefault("_rate_cache", {})
        key = (float(w), self.weight.device)
        if key not in cache:
            cache[key] = torch.tensor([float(w)], dtype=torch.float32, device=self.weight.device)
        return cache[key]

    def forward(self, x, w=1.0):
        if np.isscalar(w):
            w = self._rate_tensor(w)
        else:
            w = w.reshape(-1).to(torch.float32)
        squeeze = x.dim() == 1
        x2 = x.view(1, -1) if squeeze else x
        out = ops.sinusoidal_encoding(x2, self.weight, w)
        return out[0] if squeeze else out


class DeviceEmbedding(nn.Embedding):
    """nn.Embedding whose lookup/scatter run on the dv3b200 kernels (ids are range-checked on device)."""

    def forward(self, x):
        return ops.embedding(x, self.weight, self.padding_idx)


def Linear(in_features, out_features, dropout=0):
    """Weight-normalized Linear layer (input: N x T x C) -- reference modules.py:80-85."""
    scratch = nn.Linear(in_features, out_features)
    scratch.weight.data.normal_(mean=0, std=math.sqrt((1 - dropout) / in_features))
    return WNLinear(in_features, out_features, init_weight=scratch.weight.data,
                    init_bias=torch.zeros(out_features))


def Embedding(num_embeddings, embedding_dim, padding_idx, std=0.01):
    """reference modules.py:88-91."""
    m = DeviceEmbedding(num_embeddings, embedding_dim, padding_idx=padding_idx)
    m.weight.data.normal_(0, std)
    return m


def Conv1d(in_channels, out_channels, kernel_size, dropout=0, std_mul=4.0, **kwargs):
    """reference modules.py:94-100."""
    scratch = nn.Conv1d(in_channels, out_channels, kernel_size, **kwargs)
    std = math.sqrt((std_mul * (1.0 - dropout)) / (scratch.kernel_size[0] * in_channels))
    scratch.weight.data.normal_(mean=0, std=std)
    return _Conv1d(in_channels, out_channels, kernel_size, padding=scratch.padding[0],
                   dilation=scratch.dilation[0], init_weight=scratch.weight.data,
                   init_bias=torch.zeros(out_channels))


def ConvTranspose1d(in_channels, out_channels, kernel_size, dropout=0, std_mul=1.0, **kwargs):
    """reference modules.py:103-109."""
    scratch = nn.ConvTranspose1d(in_channels, out_channels, kernel_size, **kwargs)
    std = math.sqrt((std_mul * (1.0 - dropout)) / (scratch.kernel_size[0] * in_channels))
    scratch.weight.data.normal_(mean=0, std=std)
    return _ConvTranspose1d(in_channels, out_channels, kernel_size, padding=scratch.padding[0],
                            stride=scratch.stride[0], init_weight=scratch.weight.data,
                            init_bias=torch.zeros(out_channels))


class _GatedConv(nn.Module):
    """Shared shape logic of Conv1dGLU / HighwayConv1d: one fused kernel per block."""

    def _make_conv(self, in_channels, out_channels, kernel_size, padding, dilation, causal, dropout, std_mul):
        if in_channels != out_channels:
            raise ValueError("the fused ConvBlock needs in_channels == out_channels (true of every block "
                             "the reference builders create)")
        if padding is None:
            padding = (kernel_size - 1) * dilation if causal else (kernel_size - 1) // 2 * dilation
        self.causal = causal
        self.conv = Conv1d(in_channels, 2 * out_channels, kernel_size, dropout=dropout, padding=padding,
                           dilation=dilation, std_mul=std_mul)

    def _step(self, x, mode, spk=None, residual=False):
        """One autoregressive step of the block on x (B, T, C) (newest frame = x[:, -1]) -> (B, 1, C)."""
        if self.training:
            raise RuntimeError("incremental_forward only supports eval mode")
        from .incremental import ModuleStepper
        st = self.__dict__.get("_stepper")
        if st is None or st.B != x.size(0):
            st = self.__dict__["_stepper"] = ModuleStepper(self.conv, x.size(0), mode=mode, spk=spk,
                                                           residual=residual)
        return st.step(x[:, -1, :])

    def clear_buffer(self):
        self.__dict__.pop("_stepper", None)


class Conv1dGLU(_GatedConv):
    """(Dilated) Conv1d + gated linear unit + (optionally) speaker embedding -- reference modules.py:112-167."""

    def __init__(self, n_speakers, speaker_embed_dim, in_channels, out_channels, kernel_size, dropout,
                 padding=None, dilation=1, causal=False, residual=False, std_mul=4.0):
        super().__init__()
        self.dropout = dropout
        self.residual = residual
        self._make_conv(in_channels, out_channels, kernel_size, padding, dilation, causal, dropout, std_mul)
        self.speaker_proj = Linear(speaker_embed_dim, out_channels) if n_speakers > 1 else None

    def forward(self, x, speaker_embed=None, fuse_residual=None):
        """x (B, C, T); speaker_embed (B, T, S) time-expanded (and, in training, dropped-out) embedding.
        fuse_residual=True computes (block(x) + x)*sqrt(.5) in the kernel even when the module was built with
        residual=False -- the decoder applies exactly that outside the block when no attention layer sits in between
        (reference deepvoice3.py:333-349)."""
        spk = None
        if self.speaker_proj is not None:
            spk = F.softsign(self.speaker_proj.forward_bct(ops.transpose12(speaker_embed)))
        c = self.conv
        residual = self.residual if fuse_residual is None else bool(fuse_residual)
        return ops.convblock(x, c.weight_v, c.weight_g, c.bias, spk, c.kernel_size[0], c.dilation[0],
                             self.causal, ops.MODE_GLU, residual, self.dropout, self.training)


    def incremental_forward(self, x, speaker_embed=None):
        """reference modules.py:142-143: x (B, 1, C); speaker_embed (B, S) -- constant over the sequence, so its
        softsign projection is computed when the step state is created (clear_buffer resets it)."""
        spk = None
        if self.speaker_proj is not None and "_stepper" not in self.__dict__:
            spk = F.softsign(self.speaker_proj(speaker_embed.reshape(x.size(0), -1)))
        return self._step(x, 1, spk=spk, residual=self.residual)


class HighwayConv1d(_GatedConv):
    """Weight-normalized Conv1d + highway gate -- reference modules.py:170-229 (glu=False branch)."""

    def __init__(self, in_channels, out_channels, kernel_size=1, padding=None, dilation=1, causal=False,
                 dropout=0, std_mul=None, glu=False):
        super().__init__()
        if glu:
            raise NotImplementedError("glu=True is never used by the reference builders")
        self.dropout = dropout
        self.glu = glu
        self._make_conv(in_channels, out_channels, kernel_size, padding, dilation, causal, dropout,
                        1.0 if std_mul is None else std_mul)

    def forward(self, x):
        c = self.conv
        return ops.convblock(x, c.weight_v, c.weight_g, c.bias, None, c.kernel_size[0], c.dilation[0],
                             self.causal, ops.MODE_HIGHWAY, True, self.dropout, self.training)

    def incremental_forward(self, x):
        """reference modules.py:197-198."""
        return self._step(x, 2)


def get_mask_from_lengths(memory, memory_lengths):
    """True where the memory position is padding -- reference modules.py:232-241.
    memory: (batch, max_time, dim); memory_lengths: array like on the host (the reference's calling
    convention, train.py:643) or an int64 tensor already on memory's device (no H2D copy: graph-capture safe;
    max_time must then equal max(lengths), which the reference's masked_fill requires anyway)."""
    if torch.is_tensor(memory_lengths) and memory_lengths.device == memory.device and memory.is_cuda:
        steps = torch.arange(memory.size(1), device=memory.device)
        return steps[None, :] >= memory_lengths.view(-1, 1)
    max_len = int(max(memory_lengths))
    lengths = torch.as_tensor(np.asarray(memory_lengths)).view(-1, 1)
    mask = torch.arange(max_len).expand(memory.size(0), max_len) < lengths
    return (~mask).to(memory.device)


def run_conv_stack(layers, x, speaker_embed_btc=None, boundaries=None):
    """Run a ModuleList/Sequential of [Conv1d | ReLU | Sigmoid | ConvTranspose1d | Conv1dGLU | HighwayConv1d]
    on x (B, C, T), fusing every ``Conv1d -> ReLU`` pair into one kernel launch.
    boundaries: {layer index: tag} -- the input of that layer is an ops.grad_boundary (its gradient being ready means
    the parameter gradients of layers[index:] are final)."""
    layers = list(layers)
    i = 0
    while i < len(layers):
        f = layers[i]
        if boundaries and i in boundaries:
            x = ops.grad_boundary(x, boundaries[i])
        fuse_relu = isinstance(f, _Conv1d) and i + 1 < len(layers) and isinstance(layers[i + 1], nn.ReLU)
        if isinstance(f, _Conv1d):
            x = f(x, relu=fuse_relu)
        elif isinstance(f, Conv1dGLU):
            x = f(x, speaker_embed_btc)
        elif isinstance(f, nn.ReLU):
            x = torch.relu(x)
        else:
            x = f(x)
        i += 2 if fuse_relu else 1
    return x
