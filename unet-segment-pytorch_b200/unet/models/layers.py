"""Building blocks of the B200 U-Net, drop-in for ``unet.models.layers`` of the reference.

Every class keeps the reference's constructor signature and registers *real*
``nn.Conv2d`` / ``nn.BatchNorm2d`` / ``nn.ConvTranspose2d`` children under the
reference's attribute names and in its creation order, purely as parameter and
buffer holders: ``state_dict()`` keys / shapes / dtypes, default initialisation
(and its RNG consumption order), ``named_parameters()``, ``copy.deepcopy`` and
``.to(device)`` therefore behave exactly like the reference
(reference: unet/models/layers.py:16-255).  ``forward`` never calls those
children: it launches the fused sm_100a kernels through ``unet.ops``.

Activations travel between blocks as logical-NCHW, channels_last, bf16 tensors
(physically NHWC).  Any float NCHW tensor is accepted as input.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import fp32, ops


def _stage(x0, x1, conv: nn.Conv2d, bn: nn.BatchNorm2d, pool: bool = False):
    return ops.ConvBnRelu.apply(x0, x1, conv.weight, bn.weight, bn.bias, bn, pool)


class DoubleConv(nn.Module):
    """(conv3x3 -> BN -> ReLU) x 2.  Reference: layers.py:16-41."""

    def __init__(self, in_channels: int, out_channels: int, mid_channels: int = None):
        super().__init__()
        mid = mid_channels if mid_channels is not None else out_channels
        self.double_conv = nn.Sequential(
            nn.Conv2d(in_channels, mid, kernel_size=3, padding=1, bias=False),
            nn.BatchNorm2d(mid),
            nn.ReLU(inplace=True),
            nn.Conv2d(mid, out_channels, kernel_size=3, padding=1, bias=False),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(inplace=True),
        )

    def _run(self, x0, x1=None, pool_out: bool = False):
        if fp32.active():
            return fp32.double_conv(self, x0, x1, pool_out)
        seq = self.double_conv
        cin = x0.shape[1] + (x1.shape[1] if x1 is not None else 0)
        if cin % 16 != 0:
            # network stem: a handful of input channels, direct fp32 convolution
            if x1 is not None:
                raise RuntimeError("concatenated inputs need channel counts that are multiples of 16")
            a = ops.ConvInBnRelu.apply(x0, seq[0].weight, seq[1].weight, seq[1].bias, seq[1])
        else:
            a, _ = _stage(x0, x1, seq[0], seq[1])
        return _stage(a, None, seq[3], seq[4], pool=pool_out)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._run(x)[0]


class Down(nn.Module):
    """MaxPool2d(2) -> DoubleConv.  Reference: layers.py:44-61.

    Inside ``UNet`` the pool is produced by the previous block's epilogue pass
    (see ``UNet.forward``); standalone use pools here."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.maxpool_conv = nn.Sequential(nn.MaxPool2d(2), DoubleConv(in_channels, out_channels))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if fp32.active():
            return self.maxpool_conv[1](fp32.maxpool(x))
        return self.maxpool_conv[1](ops.MaxPool2x2.apply(x))

    def forward_pooled(self, pooled: torch.Tensor, pool_out: bool):
        """Input already pooled; returns (activation, pooled activation or None)."""
        return self.maxpool_conv[1]._run(pooled, None, pool_out)


class Up(nn.Module):
    """Upsample (or ConvTranspose2d) -> pad -> concat([skip, up]) -> DoubleConv.
    Reference: layers.py:64-106.  The concat is virtual: the conv kernel walks both tensors."""

    def __init__(self, in_channels: int, out_channels: int, bilinear: bool = True):
        super().__init__()
        if bilinear:
            self.up = nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True)
            self.conv = DoubleConv(in_channels, out_channels, in_channels // 2)
        else:
            self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
            self.conv = DoubleConv(in_channels, out_channels)

    def _upsampled(self, x1, skip):
        if fp32.active():
            if isinstance(self.up, nn.ConvTranspose2d):
                return fp32.conv_transpose2x2(self.up, x1, skip.shape[2], skip.shape[3])
            return fp32.upsample(x1, skip.shape[2], skip.shape[3])
        if isinstance(self.up, nn.ConvTranspose2d):
            return ops.conv_transpose2x2(x1, self.up.weight, self.up.bias, skip.shape[2], skip.shape[3])
        return ops.Upsample2x.apply(x1, skip.shape[2], skip.shape[3])

    def forward(self, x1: torch.Tensor, x2: torch.Tensor) -> torch.Tensor:
        return self.conv._run(x2, self._upsampled(x1, x2))[0]


class OutConv(nn.Module):
    """1x1 conv with bias to fp32 logits.  Reference: layers.py:109-123."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=1)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if fp32.active():
            return fp32.outc(self, x)
        return ops.OutConvFn.apply(x, self.conv.weight, self.conv.bias)


class _BnView:
    """What unet.ops / unet.fp32 read from a BatchNorm2d, with the channel vectors padded by `pad` neutral
    channels (gamma 1, beta 0, running statistics 0 / 1); ``write_back`` returns the real channels' running
    statistics to the module (``num_batches_tracked`` is shared and advanced in place)."""

    def __init__(self, bn: nn.BatchNorm2d, pad: int):
        self._bn, self._c = bn, bn.num_features
        self.training, self.momentum, self.eps = bn.training, bn.momentum, bn.eps
        self.track_running_stats = bn.track_running_stats
        self.weight = F.pad(bn.weight, (0, pad), value=1.0)
        self.bias = F.pad(bn.bias, (0, pad))
        self.running_mean = F.pad(bn.running_mean, (0, pad)) if bn.running_mean is not None else None
        self.running_var = F.pad(bn.running_var, (0, pad), value=1.0) if bn.running_var is not None else None
        self.num_batches_tracked = bn.num_batches_tracked

    @torch.no_grad()
    def write_back(self):
        if self.training and self.track_running_stats and self.running_mean is not None:
            self._bn.running_mean.copy_(self.running_mean[:self._c])
            self._bn.running_var.copy_(self.running_var[:self._c])


class _W:
    def __init__(self, weight):
        self.weight = weight


class _PaddedGate:
    """An AttentionGate whose inter-channel count is not a multiple of 16 (base_features=16: 8 channels), seen
    through padding: the tensor-core kernels need K and N in multiples of 16, so W_g / W_x get zero output rows,
    psi zero input columns and the two BatchNorms neutral channels.  The padded channels stay exactly zero through
    the gate (zero projection -> BatchNorm of a zero channel -> ReLU(0) -> zero psi weight), gradients reach the real
    parameters through the padding's own autograd, and the module's parameters / state_dict are untouched."""

    def __init__(self, gate: "AttentionGate", pad: int):
        self._gate = gate
        self.training = gate.training
        self.W_g = (_W(F.pad(gate.W_g[0].weight, (0, 0, 0, 0, 0, 0, 0, pad))), _BnView(gate.W_g[1], pad))
        self.W_x = (_W(F.pad(gate.W_x[0].weight, (0, 0, 0, 0, 0, 0, 0, pad))), _BnView(gate.W_x[1], pad))
        self.psi = (_W(F.pad(gate.psi[0].weight, (0, 0, 0, 0, 0, pad))), gate.psi[1])

    def parameters(self):
        return self._gate.parameters()

    def write_back(self):
        self.W_g[1].write_back()
        self.W_x[1].write_back()


class AttentionGate(nn.Module):
    """Additive attention gate.  Reference: layers.py:126-192."""

    def __init__(self, gate_channels: int, skip_channels: int, inter_channels: int = None):
        super().__init__()
        inter = inter_channels if inter_channels is not None else skip_channels // 2
        self.W_g = nn.Sequential(nn.Conv2d(gate_channels, inter, kernel_size=1, bias=False),
                                 nn.BatchNorm2d(inter))
        self.W_x = nn.Sequential(nn.Conv2d(skip_channels, inter, kernel_size=1, bias=False),
                                 nn.BatchNorm2d(inter))
        self.psi = nn.Sequential(nn.Conv2d(inter, 1, kernel_size=1, bias=False), nn.BatchNorm2d(1),
                                 nn.Sigmoid())
        self.relu = nn.ReLU(inplace=True)

    def forward(self, g: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        inter = self.W_g[0].weight.shape[0]
        if inter % 16 != 0:
            if inter % 8 != 0:
                raise RuntimeError("AttentionGate needs an inter-channel count that is a multiple of 8")
            view = _PaddedGate(self, 16 - inter % 16)
            out = self._gate(view, g, x)
            view.write_back()
            return out
        return self._gate(self, g, x)

    @staticmethod
    def _gate(m, g, x):
        if fp32.active():
            return fp32.gate(m, g, x)
        bg, bx, bp = m.W_g[1], m.W_x[1], m.psi[1]
        return ops.AttentionGateFn.apply(g, x, m.W_g[0].weight, m.W_x[0].weight, m.psi[0].weight,
                                         bg.weight, bg.bias, bx.weight, bx.bias, bp.weight, bp.bias,
                                         bg, bx, bp)


class AttentionUp(nn.Module):
    """Gate the skip with the un-upsampled decoder tensor, then Up.  Reference: layers.py:195-255."""

    def __init__(self, in_channels: int, out_channels: int, bilinear: bool = True):
        super().__init__()
        if bilinear:
            self.up = nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True)
            gate_channels = in_channels // 2
            self.conv = DoubleConv(in_channels, out_channels, in_channels // 2)
        else:
            self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
            gate_channels = in_channels
            self.conv = DoubleConv(in_channels, out_channels)
        self.attention = AttentionGate(gate_channels=gate_channels, skip_channels=in_channels // 2)

    _upsampled = Up._upsampled

    def forward(self, x1: torch.Tensor, x2: torch.Tensor) -> torch.Tensor:
        gated = self.attention(x1, x2)
        return self.conv._run(gated, self._upsampled(x1, gated))[0]
