"""StyleGAN (v1) generator: parameter layout + the CUDA-backed mapping network.

Mirror of the module tree of /root/reference/models/stylegan/model.py:26-389 (``StyleGAN_G``): same sub-module names (so
``named_modules()`` / layer validation / ``stylegan_{class}_{res}.pt`` state dicts line up) and the same parameter creation
order and expressions (so ``torch.manual_seed(s)`` followed by ``StyleGAN_G(resolution)`` gives the reference's random init
bit-for-bit).  As in the reference, one LeakyReLU instance is shared by all layers of G_mapping and one by all epilogues of
G_synthesis, so ``named_modules()`` lists each only under its first name.

One G_mapping layer (model.py:26-49, :190-216) is
    lrelu_0.2( x (W w_mul)^T + b_mul b ),   w_mul = sqrt(2)/sqrt(512) * 0.01,  b_mul = 0.01,
and the packed StyleGAN2 mapping kernels compute sqrt(2) lrelu_0.2( x (W 0.01/sqrt(512))^T + 0.01 b' ).  Leaky-ReLU is
positively homogeneous, so the two are equal for b' = b / sqrt(2): G_mapping runs as ``PackedMapping(W, b/sqrt(2), 0.01)``
behind the same PixelNorm (eps 1e-8 in both).

The synthesis network runs as one C-ABI call (csrc/synthesis_sg1.cu) driven by ``models.wrappers.StyleGAN``; its modules hold
the parameters in the reference's layout and give the hooks their names.  The ones whose output is a stop point of the fused
chain (blocks, LayerEpilogue, StyleMod, StyleMod.lin, the convs, torgb, G_synthesis) are called with ``_result=`` to hand that
output to their hooks; the others (noise, activation, instance_norm, upscale, blur) have no stand-alone forward.
"""
from __future__ import annotations

import math
from collections import OrderedDict

import numpy as np
import torch
from torch import nn

from .. import _native

DLATENT = 512
N_MAPPING = 8
MAPPING_LR = 0.01


class _NotBuilt(nn.Module):
    def forward(self, *a, **k):
        raise NotImplementedError(
            f"StyleGAN {self.__class__.__name__} has no stand-alone forward: the synthesis network runs as one fused C-ABI call "
            "(StyleGAN.forward / partial_forward); there is no PyTorch/CPU fallback")


class _StopPoint(nn.Module):
    """A module whose output is a stop point of the fused synthesis chain: ``forward(_result=t)`` hands ``t`` to its hooks."""

    def forward(self, *a, _result=None, **k):
        if _result is None:
            raise NotImplementedError(
                f"StyleGAN {self.__class__.__name__} runs inside the fused synthesis chain (StyleGAN.forward / partial_forward); "
                "there is no PyTorch/CPU fallback")
        return _result


class MyLinear(nn.Module):
    """model.py:26-49.  Parameter holder; ``forward`` (a g_mapping dense layer run on its own, when a g_mapping child is
    hooked) is the native fp32 linear kernel."""

    def __init__(self, input_size, output_size, gain=2 ** 0.5, use_wscale=False, lrmul=1, bias=True):
        super().__init__()
        he_std = gain * input_size ** (-0.5)
        if use_wscale:
            init_std = 1.0 / lrmul
            self.w_mul = he_std * lrmul
        else:
            init_std = he_std / lrmul
            self.w_mul = lrmul
        self.weight = nn.Parameter(torch.randn(output_size, input_size) * init_std)
        if bias:
            self.bias = nn.Parameter(torch.zeros(output_size))
            self.b_mul = lrmul
        else:
            self.bias = None

    def forward(self, x=None, _result=None):
        if _result is not None:                    # StyleMod.lin: the style vector computed inside the synthesis chain
            return _result
        bias = None if self.bias is None else (self.bias * self.b_mul).detach()
        return _native.linear(x, (self.weight * self.w_mul).detach(), bias)


class MyConv2d(_StopPoint):
    """model.py:51-104 (parameter holder)."""

    def __init__(self, input_channels, output_channels, kernel_size, gain=2 ** 0.5, use_wscale=False, lrmul=1, bias=True,
                 intermediate=None, upscale=False):
        super().__init__()
        self.upscale = Upscale2d() if upscale else None
        he_std = gain * (input_channels * kernel_size ** 2) ** (-0.5)
        self.kernel_size = kernel_size
        if use_wscale:
            init_std = 1.0 / lrmul
            self.w_mul = he_std * lrmul
        else:
            init_std = he_std / lrmul
            self.w_mul = lrmul
        self.weight = nn.Parameter(torch.randn(output_channels, input_channels, kernel_size, kernel_size) * init_std)
        if bias:
            self.bias = nn.Parameter(torch.zeros(output_channels))
            self.b_mul = lrmul
        else:
            self.bias = None
        self.intermediate = intermediate


class NoiseLayer(_NotBuilt):
    """model.py:106-122: per-channel weight times a per-pixel map (``noise``, set by StyleGAN.set_noise_seed)."""

    def __init__(self, channels):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(channels))
        self.noise = None


class StyleMod(_StopPoint):
    """model.py:124-136."""

    def __init__(self, latent_size, channels, use_wscale):
        super().__init__()
        self.lin = MyLinear(latent_size, channels * 2, gain=1.0, use_wscale=use_wscale)


class PixelNormLayer(nn.Module):
    """model.py:138-143: x * rsqrt(mean(x^2) + 1e-8) over the feature axis (the CUDA PixelNorm kernel)."""

    def __init__(self, epsilon=1e-8):
        super().__init__()
        self.epsilon = epsilon

    def forward(self, x):
        return _native.mapping_pixelnorm(x)


class LeakyReLU(nn.Module):
    """nn.LeakyReLU(0.2) of model.py:192-193 / :332-333 (no gain); the CUDA elementwise kernel."""

    def __init__(self, negative_slope=0.2):
        super().__init__()
        self.negative_slope = negative_slope

    def forward(self, x):
        return _native.leaky_relu(x, self.negative_slope)


class InstanceNorm2d(_NotBuilt):
    """nn.InstanceNorm2d(channels) of model.py:241: eps 1e-5, no affine parameters, no running statistics."""

    def __init__(self, num_features, eps=1e-5):
        super().__init__()
        self.num_features, self.eps = num_features, eps


class BlurLayer(_NotBuilt):
    """model.py:145-169: [1,2,1] x [1,2,1] / 16, pad 1."""

    def __init__(self, kernel=(1, 2, 1), normalize=True, flip=False, stride=1):
        super().__init__()
        kernel = torch.tensor([1, 2, 1], dtype=torch.float32)
        kernel = kernel[:, None] * kernel[None, :]
        kernel = kernel[None, None]
        if normalize:
            kernel = kernel / kernel.sum()
        if flip:
            kernel = torch.flip(kernel, [2, 3])
        self.register_buffer("kernel", kernel)
        self.stride = stride


class Upscale2d(_NotBuilt):
    """model.py:171-188: nearest-neighbour x2."""

    def __init__(self, factor=2, gain=1):
        super().__init__()
        assert isinstance(factor, int) and factor >= 1
        self.gain, self.factor = gain, factor


class G_mapping(nn.Sequential):
    """model.py:190-216: children 'pixel_norm', 'dense0' .. 'dense7' and 'dense0_act' .. 'dense7_act' (one shared module).

    forward() runs the whole network in one C-ABI call unless a child carries a hook, in which case the children run one
    by one (PixelNorm kernel, fp32 linear kernel, leaky-ReLU kernel) so that the hooks fire and their edits propagate."""

    def __init__(self, nonlinearity="lrelu", use_wscale=True):
        if nonlinearity != "lrelu":
            raise NotImplementedError("G_mapping: only the 'lrelu' nonlinearity (the reference's default) is built")
        act, gain = LeakyReLU(negative_slope=0.2), np.sqrt(2)
        layers = [("pixel_norm", PixelNormLayer())]
        for i in range(N_MAPPING):
            layers.append((f"dense{i}", MyLinear(DLATENT, DLATENT, gain=gain, lrmul=MAPPING_LR, use_wscale=use_wscale)))
            layers.append((f"dense{i}_act", act))
        super().__init__(OrderedDict(layers))
        self._packed = None
        self._packed_key = None

    def dense_layers(self):
        return [getattr(self, f"dense{i}") for i in range(N_MAPPING)]

    def packed(self) -> "_native.PackedMapping":
        """The eight layers for the fused mapping kernels, b' = b / sqrt(2) (see the module docstring); re-packed when a
        parameter changes."""
        lins = self.dense_layers()
        key = tuple((l.weight._version, l.bias._version, l.weight.data_ptr(), l.bias.data_ptr()) for l in lins)
        if self._packed is None or self._packed_key != key:
            w = torch.stack([l.weight.detach() for l in lins])
            b = torch.stack([l.bias.detach() for l in lins]) / math.sqrt(2.0)
            self._packed = _native.PackedMapping(w, b, MAPPING_LR)
            self._packed_key = key
        return self._packed

    def forward(self, x):
        if any(len(m._forward_hooks) or len(m._forward_pre_hooks) for m in self.modules() if m is not self):
            # the shared activation module is called under each of its eight names, as in the reference
            x = self.pixel_norm(x)
            for lin in self.dense_layers():
                x = self.dense0_act(lin(x))
            return x
        return self.packed().forward(x, pixelnorm=True)


class LayerEpilogue(_StopPoint):
    """model.py:230-253 (parameter holder): top_epi.{noise, activation, instance_norm}, style_mod.lin."""

    def __init__(self, channels, dlatent_size, use_wscale, use_noise, use_pixel_norm, use_instance_norm, use_styles,
                 activation_layer):
        super().__init__()
        if use_pixel_norm:
            raise NotImplementedError("LayerEpilogue: use_pixel_norm is not built (the reference's G_synthesis default is False)")
        layers = []
        if use_noise:
            layers.append(("noise", NoiseLayer(channels)))
        layers.append(("activation", activation_layer))
        if use_instance_norm:
            layers.append(("instance_norm", InstanceNorm2d(channels)))
        self.top_epi = nn.Sequential(OrderedDict(layers))
        self.style_mod = StyleMod(dlatent_size, channels, use_wscale=use_wscale) if use_styles else None


class InputBlock(_StopPoint):
    """model.py:256-281 (parameter holder): const, bias, epi1, conv, epi2."""

    def __init__(self, nf, dlatent_size, const_input_layer, gain, use_wscale, use_noise, use_pixel_norm, use_instance_norm,
                 use_styles, activation_layer):
        super().__init__()
        if not const_input_layer:
            raise NotImplementedError("InputBlock: only the learned-constant input (the reference's default) is built")
        self.const_input_layer = const_input_layer
        self.nf = nf
        self.const = nn.Parameter(torch.ones(1, nf, 4, 4))
        self.bias = nn.Parameter(torch.ones(nf))
        self.epi1 = LayerEpilogue(nf, dlatent_size, use_wscale, use_noise, use_pixel_norm, use_instance_norm, use_styles,
                                  activation_layer)
        self.conv = MyConv2d(nf, nf, 3, gain=gain, use_wscale=use_wscale)
        self.epi2 = LayerEpilogue(nf, dlatent_size, use_wscale, use_noise, use_pixel_norm, use_instance_norm, use_styles,
                                  activation_layer)


class GSynthesisBlock(_StopPoint):
    """model.py:284-303 (parameter holder): conv0_up (with upscale and blur children), epi1, conv1, epi2."""

    def __init__(self, in_channels, out_channels, blur_filter, dlatent_size, gain, use_wscale, use_noise, use_pixel_norm,
                 use_instance_norm, use_styles, activation_layer):
        super().__init__()
        blur = BlurLayer(blur_filter) if blur_filter else None
        self.conv0_up = MyConv2d(in_channels, out_channels, kernel_size=3, gain=gain, use_wscale=use_wscale,
                                 intermediate=blur, upscale=True)
        self.epi1 = LayerEpilogue(out_channels, dlatent_size, use_wscale, use_noise, use_pixel_norm, use_instance_norm,
                                  use_styles, activation_layer)
        self.conv1 = MyConv2d(out_channels, out_channels, kernel_size=3, gain=gain, use_wscale=use_wscale)
        self.epi2 = LayerEpilogue(out_channels, dlatent_size, use_wscale, use_noise, use_pixel_norm, use_instance_norm,
                                  use_styles, activation_layer)


class G_synthesis(_StopPoint):
    """model.py:305-363 (parameter holder) with the reference's defaults: blocks '4x4' .. 'RxR', torgb."""

    def __init__(self, dlatent_size=DLATENT, num_channels=3, resolution=1024, fmap_base=8192, fmap_decay=1.0, fmap_max=512,
                 use_styles=True, const_input_layer=True, use_noise=True, nonlinearity="lrelu", use_wscale=True,
                 use_pixel_norm=False, use_instance_norm=True, blur_filter=(1, 2, 1)):
        super().__init__()

        def nf(stage):
            return min(int(fmap_base / (2.0 ** (stage * fmap_decay))), fmap_max)
        self.dlatent_size = dlatent_size
        resolution_log2 = int(np.log2(resolution))
        assert resolution == 2 ** resolution_log2 and resolution >= 4
        if nonlinearity != "lrelu":
            raise NotImplementedError("G_synthesis: only the 'lrelu' nonlinearity (the reference's default) is built")
        act, gain = LeakyReLU(negative_slope=0.2), np.sqrt(2)
        blocks, last_channels = [], None
        for res in range(2, resolution_log2 + 1):
            channels = nf(res - 1)
            name = f"{2 ** res}x{2 ** res}"
            if res == 2:
                blocks.append((name, InputBlock(channels, dlatent_size, const_input_layer, gain, use_wscale, use_noise,
                                                use_pixel_norm, use_instance_norm, use_styles, act)))
            else:
                blocks.append((name, GSynthesisBlock(last_channels, channels, list(blur_filter), dlatent_size, gain,
                                                     use_wscale, use_noise, use_pixel_norm, use_instance_norm, use_styles, act)))
            last_channels = channels
        self.torgb = MyConv2d(channels, num_channels, 1, gain=1, use_wscale=use_wscale)
        self.blocks = nn.ModuleDict(OrderedDict(blocks))


class StyleGAN_G(nn.Sequential):
    """model.py:366-389: children 'g_mapping' and 'g_synthesis'."""

    def __init__(self, resolution, truncation=1.0):
        self.resolution = resolution
        super().__init__(OrderedDict([("g_mapping", G_mapping()), ("g_synthesis", G_synthesis(resolution=resolution))]))

    def forward(self, x, latent_is_w=False):
        raise NotImplementedError("StyleGAN_G.forward: images come from the wrapper's fused synthesis chain (StyleGAN.forward); "
                                  "there is no PyTorch/CPU fallback")
