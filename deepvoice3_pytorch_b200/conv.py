"""Weight-normalised Conv1d / ConvTranspose1d / Linear parameter holders.

Mirrors the objects the reference gets from ``nn.utils.weight_norm(conv.Conv1d(...))``
(reference deepvoice3_pytorch/conv.py:7-15 + modules.py:94-100): parameters are named ``bias``,
``weight_g`` and ``weight_v`` with the reference's shapes, so reference checkpoints load key-for-key.
The arithmetic (w = g*v/||v||, the convolution, its gradients) runs in csrc/ through ops.py.
"""
import torch
from torch import nn

from . import ops


class _WeightNormed(nn.Module):
    def _set_params(self, weight, bias):
        """weight: the un-normalised init tensor; g starts at ||v|| so that w == weight (weight_norm dim=0)."""
        self.bias = nn.Parameter(bias)
        norm = torch.norm_except_dim(weight, 2, 0)      # bit-identical to weight_norm's initial g
        self.weight_g = nn.Parameter(norm)
        self.weight_v = nn.Parameter(weight)

    @property
    def weight(self):
        """The effective weight, for inspection (computed with torch; not on the hot path)."""
        v, g = self.weight_v, self.weight_g
        return g * v / v.pow(2).sum(tuple(range(1, v.dim())), keepdim=True).sqrt()


class Conv1d(_WeightNormed):
    """Dilated 1-D convolution, (B, Cin, T) -> (B, Cout, T).  ``padding`` must be the 'same' padding
    (k-1)//2*dilation or the causal padding (k-1)*dilation whose future half the caller trims
    (reference modules.py:126,155) -- the kernel pads on the left only instead of trimming."""

    def __init__(self, in_channels, out_channels, kernel_size, padding=0, dilation=1, init_weight=None,
                 init_bias=None):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.dilation, self.padding = (kernel_size,), (dilation,), (padding,)
        k, d = kernel_size, dilation
        if padding == (k - 1) // 2 * d:
            self.causal_padding = False
        elif padding == (k - 1) * d:
            self.causal_padding = True
        else:
            raise ValueError("unsupported padding %d for kernel_size %d dilation %d" % (padding, k, d))
        w = init_weight if init_weight is not None else torch.zeros(out_channels, in_channels, k)
        b = init_bias if init_bias is not None else torch.zeros(out_channels)
        self._set_params(w, b)

    def forward(self, x, relu=False, causal=None):
        """causal=None: treat causal padding like the reference does (output length T + (k-1)d is not
        produced; callers of the causal form always trim to T, which is what the kernel computes)."""
        causal = self.causal_padding if causal is None else causal
        return ops.conv1d(x, self.weight_v, self.weight_g, self.bias, self.kernel_size[0], self.dilation[0],
                          causal=causal, relu=relu)

    def incremental_forward(self, input):
        """input (B, T, Cin): the newest frame input[:, -1] enters the ring buffer of the last (k-1)*dilation+1
        frames -> (B, 1, Cout) (reference conv.py:17-46).  Eval mode only; ``clear_buffer`` starts a new sequence
        (and re-folds the weight norm)."""
        if self.training:
            raise RuntimeError("incremental_forward only supports eval mode")
        from .incremental import ModuleStepper
        st = self.__dict__.get("_stepper")
        if st is None or st.B != input.size(0):
            st = self.__dict__["_stepper"] = ModuleStepper(self, input.size(0))
        return st.step(input[:, -1, :])

    def clear_buffer(self):
        self.__dict__.pop("_stepper", None)

    def extra_repr(self):
        return "%d, %d, kernel_size=%d, dilation=%d, padding=%d" % (
            self.in_channels, self.out_channels, self.kernel_size[0], self.dilation[0], self.padding[0])


class ConvTranspose1d(_WeightNormed):
    """kernel_size=2, stride=2 time upsampler, (B, Cin, T) -> (B, Cout, 2T); weight_v (Cin, Cout, 2),
    normalised over dim 0 = Cin exactly like weight_norm on nn.ConvTranspose1d (reference modules.py:103-109)."""

    def __init__(self, in_channels, out_channels, kernel_size, padding=0, stride=2, init_weight=None,
                 init_bias=None):
        super().__init__()
        if not (kernel_size == 2 and stride == 2 and padding == 0):
            raise ValueError("only kernel_size=2, stride=2, padding=0 is supported (all the builders use)")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding = (2,), (2,), (0,)
        w = init_weight if init_weight is not None else torch.zeros(in_channels, out_channels, 2)
        b = init_bias if init_bias is not None else torch.zeros(out_channels)
        self._set_params(w, b)

    def forward(self, x):
        return ops.conv_transpose1d_k2s2(x, self.weight_v, self.weight_g, self.bias)


class WNLinear(_WeightNormed):
    """Weight-normed nn.Linear over the last dim; weight_v (out, in), weight_g (out, 1)."""

    def __init__(self, in_features, out_features, init_weight=None, init_bias=None):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        w = init_weight if init_weight is not None else torch.zeros(out_features, in_features)
        b = init_bias if init_bias is not None else torch.zeros(out_features)
        self._set_params(w, b)

    def forward(self, x):
        return ops.linear(x, self.weight_v, self.weight_g, self.bias)

    def forward_bct(self, x, relu=False):
        """Same map applied to a channel-major (B, in, T) tensor -> (B, out, T): a 1x1 conv."""
        return ops.conv1d(x, self.weight_v.view(self.out_features, self.in_features, 1),
                          self.weight_g.view(self.out_features, 1, 1), self.bias, 1, 1, relu=relu)
