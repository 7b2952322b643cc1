"""Embedding CNNs (MinAtar single-conv net, Nature-DQN three-conv net).

Constructor arguments and ``model.<i>`` parameter names match the reference
(prism/agents/models/minatar_cnn_model.py:7-46, atari_cnn_model.py:7-59).  The MinAtar embedding runs on
csrc/conv.cu; the Nature-DQN convolutions stay on cuDNN through PyTorch.
"""
import functools
import math

import torch
import torch.nn as nn


@torch.no_grad()
def _sparse_conv_init(net, p_zero):
    """Per output channel: uniform(+-1/sqrt(fan_in)) weights with ceil(p*fan_in) random zeros, zero bias."""
    for conv in (m for m in net if isinstance(m, nn.Conv2d)):
        conv.bias.zero_()
        w = conv.weight
        fan_in = w[0].numel()
        bound = math.sqrt(1.0 / fan_in)
        w.uniform_(-bound, bound)
        n_zero = int(math.ceil(p_zero * fan_in))
        flat = w.view(w.shape[0], fan_in)
        for c in range(w.shape[0]):
            flat[c, torch.randperm(fan_in)[:n_zero]] = 0.0


@functools.lru_cache(maxsize=None)
def _conv_kernel_supports(H, W, C, OC):
    from ... import _lib
    return bool(_lib.load().pb_conv3x3_relu_supported(H, W, C, OC))


def _conv_kernel_takes(hwc, conv):
    """A (H, W, C) frame goes through the conv kernel: its channels match the layer (a mismatch takes nn.Conv2d, which
    reports it) and pb_conv3x3_relu_supported accepts the shape."""
    H, W, C = (int(s) for s in hwc)
    return C == conv.in_channels and _conv_kernel_supports(H, W, C, conv.out_channels)


def _probe_dim(net, *shape):
    with torch.no_grad():
        return net(torch.zeros(1, *shape)).numel()


class MinAtarModel(nn.Module):
    """On CUDA, conv + bias + ReLU + flatten run as one kernel (``ops.conv3x3_relu_flatten``) whenever
    ``pb_conv3x3_relu_supported`` accepts the frame (C <= 14 for 10x10 frames).  Other frames take ``self.model`` on
    cuDNN, with cuDNN's TF32 path switched off process-wide at construction, as in ``NatureAtariCnn``: the backward
    runs later in the autograd engine, so a context manager around ``forward`` would not cover it, and TF32 (~1e-3)
    would miss the fp32 accuracy that the kernel and the reference hold."""

    def __init__(self, in_channels, act_fn=nn.ReLU, device="cpu", use_layer_norm=False, sparse_init_p=0.0):
        super().__init__()
        net = nn.Sequential(nn.Conv2d(in_channels, 16, kernel_size=3, stride=1), act_fn(), nn.Flatten())
        self.output_dim = _probe_dim(net, in_channels, 10, 10)
        if sparse_init_p > 0:
            _sparse_conv_init(net, sparse_init_p)
        self.model = net.to(device)
        torch.backends.cudnn.allow_tf32 = False

    def forward(self, x):
        # MinAtar observations are channels-last (10, 10, C)
        conv = self.model[0]
        if x.is_cuda and isinstance(self.model[1], nn.ReLU) and x.dim() == 4 and _conv_kernel_takes(x.shape[1:], conv):
            from .. import ops
            return ops.conv3x3_relu_flatten(x.float(), conv.weight, conv.bias)   # conv+bias+ReLU+flatten: one launch
        return self.model(x.permute(0, 3, 1, 2).float())

    def log(self, logger):
        pass


class NatureAtariCnn(nn.Module):
    _CONVS = ((32, 8, 4), (64, 4, 2), (64, 3, 1))   # (out_channels, kernel, stride)
    _LN_SHAPES = (None, (32, 20, 20), (64, 9, 9))  # LayerNorm in front of conv 2 and 3

    def __init__(self, frame_stack, feature_dim=512, act_fn=nn.ReLU, device="cpu", channels_first=True,
                 use_layer_norm=False, logger=None, sparse_init_p=0.0):
        super().__init__()
        self.channels_first = channels_first
        mods, c_in = [], frame_stack
        for (c_out, k, s), ln_shape in zip(self._CONVS, self._LN_SHAPES):
            if use_layer_norm and ln_shape is not None:
                mods.append(nn.LayerNorm(normalized_shape=ln_shape))
            mods += [nn.Conv2d(c_in, c_out, kernel_size=k, stride=s), act_fn()]
            c_in = c_out
        net = nn.Sequential(*mods, nn.Flatten())
        self.output_dim = _probe_dim(net, frame_stack, 84, 84)
        if sparse_init_p > 0:
            _sparse_conv_init(net, sparse_init_p)
        self.model = net.to(device)
        # The reference computes in fp32 and parity is judged at 1e-4 on losses and gradients: cuDNN must stay off its
        # TF32 path, forward AND backward (the backward pass runs later, inside the autograd engine, so this is the
        # process-wide switch rather than a context manager around forward).
        torch.backends.cudnn.allow_tf32 = False

    def forward(self, x):
        return self.model(x if self.channels_first else x.transpose(1, -1))

    def log(self, logger):
        pass
