"""Inference-time execution plan for the truncated torchvision ResNet50 (SURVEY 8(f) n1, the step before the path).

In eval mode a BatchNorm2d is a per-channel affine map with constants, so `bn(conv(x))` is one convolution with scaled
weights and a bias, and the ReLU (and, at the end of a bottleneck, the residual add) behind it is an epilogue cuDNN fuses
into that convolution (`cudnn_convolution_relu`, `cudnn_convolution_add_relu`). The reference executes them as separate
kernels (torchvision's Bottleneck.forward; Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:37-46 just calls the children):
on a B200 69 % of the fp32 channels_last encoder's time at batch 256 is those element-wise passes
(`bn_fw_inf` 37 %, ReLU 15 %, residual add 12 %, max-pool 5 %; profiles/r01w_launch_shares.txt), all HBM-bound.

The plan keeps every convolution but the stem's on cuDNN, and the module's parameters untouched. The stem (conv1 + bn1 +
relu + maxpool) of an fp32 plan with TF32 convolutions allowed is one kernel of the library (gh_stem_conv_pool_nhwc);
elsewhere it is the space-to-depth chain below. Folded weight copies are built lazily
from the live parameters / running statistics, and rebuilt whenever any of them changes (in-place update, load_state_dict,
.to(): detected through tensor versions and storage addresses). It is used only when the result is the same function --
module in eval mode, gradients disabled, every BatchNorm tracking running statistics -- and only for the structure it
knows (stem + Bottleneck stages); anything else runs the children one by one as before.
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

# cuDNN has no good NHWC kernel for the stem's 3-channel 7x7 stride-2 convolution (an sm80 implicit GEMM without shared
# memory: 1.33 ms of a 7.0 ms step at batch 256). The same convolution over the 2x2 space-to-depth image -- 4x4, stride
# 1, 12 channels padded to 16 -- runs on its regular tensor-core kernels in 0.58 ms (tools/time_stem.py; identical sums
# in another order: 3e-6). GRAMHEAD_STEM_S2D=0 keeps the direct convolution.
STEM_SPACE_TO_DEPTH = os.environ.get("GRAMHEAD_STEM_S2D", "1") != "0"


def _stem_space_to_depth_weight(weight: torch.Tensor) -> torch.Tensor:
    """(O, 3, 7, 7) -> (O, 16, 4, 4), channels_last: tap i' = i + 1 = 2a + r of an 8x8 kernel whose first row and column
    are zero goes to tap a of channel c*4 + r*2 + s (see gh_stem_space_to_depth)."""
    o = weight.shape[0]
    w8 = weight.new_zeros((o, 3, 8, 8))
    w8[:, :, 1:, 1:] = weight
    w12 = w8.view(o, 3, 4, 2, 4, 2).permute(0, 1, 3, 5, 2, 4).reshape(o, 12, 4, 4)
    w16 = weight.new_zeros((o, 16, 4, 4))
    w16[:, :12] = w12
    return w16.contiguous(memory_format=torch.channels_last)


def _tf32_round(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> nearest tf32 (ties away from zero), as cvt.rna.tf32.f32 rounds the image side of the fused stem."""
    bits = (x.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF) + 0x1000
    bits = bits & 0xFFFFE000
    return torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32).view(torch.float32)


def pack_stem_weight(w16: torch.Tensor) -> torch.Tensor:
    """(64, 16, 4, 4) space-to-depth stem weights -> the B operands of gh_stem_conv_pool_nhwc in its shared-memory
    layout, rounded to tf32: [tap a*4+b][half h][k-chunk q][out channel n][e] = w16[n, (2h + q)*4 + e, a, b]."""
    w = _tf32_round(w16.float().contiguous())
    return w.view(64, 2, 2, 4, 4, 4).permute(4, 5, 1, 2, 0, 3).contiguous().view(-1)


def _fold(conv: nn.Conv2d, bn: nn.BatchNorm2d, dtype: torch.dtype, channels_last: bool):
    """conv -> bn (eval) as (weight, bias, stride, padding, dilation, groups); folded in fp32, then cast."""
    var, mean = bn.running_var.detach().float(), bn.running_mean.detach().float()
    gamma = bn.weight.detach().float() if bn.weight is not None else torch.ones_like(var)
    beta = bn.bias.detach().float() if bn.bias is not None else torch.zeros_like(var)
    scale = gamma * torch.rsqrt(var + bn.eps)
    weight = conv.weight.detach().float() * scale.view(-1, 1, 1, 1)
    bias = beta - mean * scale
    if conv.bias is not None:
        bias = bias + conv.bias.detach().float() * scale
    weight = weight.to(dtype).contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    return weight, bias.to(dtype).contiguous(), conv.stride, conv.padding, conv.dilation, conv.groups


def _foldable(conv, bn) -> bool:
    return (isinstance(conv, nn.Conv2d) and type(bn) is nn.BatchNorm2d and bn.track_running_stats
            and bn.running_mean is not None and bn.running_var is not None and conv.padding_mode == "zeros"
            and not isinstance(conv.padding, str))


def _is_bottleneck(block) -> bool:
    names = ("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "relu", "downsample")
    if type(block).__name__ != "Bottleneck" or not all(hasattr(block, n) for n in names):
        return False
    if not isinstance(block.relu, nn.ReLU):
        return False
    ok = _foldable(block.conv1, block.bn1) and _foldable(block.conv2, block.bn2) and _foldable(block.conv3, block.bn3)
    if block.downsample is not None:
        ds = block.downsample
        ok = ok and isinstance(ds, nn.Sequential) and len(ds) == 2 and _foldable(ds[0], ds[1])
    return ok


def encoder_signature(encoder: nn.Module) -> Optional[Tuple]:
    """Changes whenever a parameter or buffer of the encoder is modified, replaced or moved. None when the tensors
    carry no version counter (created under torch.inference_mode()): the plan is then not used at all."""
    try:
        return tuple((t.data_ptr(), t._version) for t in list(encoder.parameters()) + list(encoder.buffers()))
    except RuntimeError:
        return None


class FoldedEncoder:
    """Callable plan: x -> (last activation, [stage activations]) like _TruncatedGramAttentionBase._run_encoder."""

    def __init__(self, stem, pool, stages, signature, dtype, channels_last):
        self.stem, self.pool, self.stages = stem, pool, stages
        self.stem_s2d = None
        self.stem_packed = None        # tf32 B operands of the fused stem kernel (fp32 plans)
        self._stem_fused = True        # A/B switch for tools/time_stem.py; the chain runs where the fused kernel does not apply
        self.signature, self.dtype, self.channels_last = signature, dtype, channels_last

    @staticmethod
    def supported(encoder: nn.Sequential) -> bool:
        if len(encoder) < 4:
            return False
        if not (_foldable(encoder[0], encoder[1]) and isinstance(encoder[2], nn.ReLU) and isinstance(encoder[3], nn.MaxPool2d)):
            return False
        for stage in list(encoder)[4:]:
            if not isinstance(stage, nn.Sequential) or not all(_is_bottleneck(b) for b in stage):
                return False
        return True

    @classmethod
    def build(cls, encoder: nn.Sequential, dtype: torch.dtype, channels_last: bool) -> Optional["FoldedEncoder"]:
        if not cls.supported(encoder):
            return None
        with torch.no_grad():
            stem = _fold(encoder[0], encoder[1], dtype, channels_last)
            conv1 = encoder[0]
            stem_s2d = None
            if (STEM_SPACE_TO_DEPTH and channels_last and conv1.in_channels == 3 and conv1.kernel_size == (7, 7)
                    and conv1.stride == (2, 2) and conv1.padding == (3, 3) and conv1.dilation == (1, 1) and conv1.groups == 1):
                stem_s2d = (_stem_space_to_depth_weight(stem[0].float()).to(dtype), stem[1], (1, 1), (0, 0), (1, 1), 1)
            stages: List[list] = []
            for stage in list(encoder)[4:]:
                blocks = []
                for b in stage:
                    c3 = _fold(b.conv3, b.bn3, dtype, channels_last)
                    down = None
                    if b.downsample is not None:
                        # relu(conv3(y) + b3 + conv_d(x) + b_d): both biases go into the fused epilogue of conv3, so the
                        # shortcut convolution needs no bias pass over its (B, 4*planes, H, W) output
                        dw, db, *geom = _fold(b.downsample[0], b.downsample[1], torch.float32, channels_last)
                        bias3 = (c3[1].float() + db).to(dtype)
                        c3 = (c3[0], bias3) + tuple(c3[2:])
                        down = (dw.to(dtype).contiguous(memory_format=torch.channels_last if channels_last
                                                        else torch.contiguous_format), None) + tuple(geom)
                    blocks.append((_fold(b.conv1, b.bn1, dtype, channels_last), _fold(b.conv2, b.bn2, dtype, channels_last),
                                   c3, down))
                stages.append(blocks)
        plan = cls(stem, encoder[3], stages, encoder_signature(encoder), dtype, channels_last)
        plan.stem_s2d = stem_s2d
        pool = encoder[3]
        if (stem_s2d is not None and dtype == torch.float32 and conv1.out_channels == 64
                and pool.kernel_size in (3, (3, 3)) and pool.stride in (2, (2, 2)) and pool.padding in (1, (1, 1))
                and pool.dilation in (1, (1, 1)) and not pool.ceil_mode and not pool.return_indices):
            plan.stem_packed = pack_stem_weight(stem_s2d[0])
        return plan

    @staticmethod
    def _conv_relu(x, p):
        w, b, stride, padding, dilation, groups = p
        return torch.cudnn_convolution_relu(x, w, b, stride, padding, dilation, groups)

    def _pool(self, x):
        p = self.pool
        k, s, pad = p.kernel_size, p.stride, p.padding
        plain = (isinstance(k, int) and isinstance(s, int) and isinstance(pad, int) and p.dilation == 1
                 and not p.ceil_mode and not p.return_indices)
        vec = 4 if x.dtype == torch.float32 else 8
        if plain and self.channels_last and x.shape[1] % vec == 0 and x.is_contiguous(memory_format=torch.channels_last):
            return ops.maxpool2d_nhwc(x, k, s, pad)
        return p(x)

    def _fused_stem_applies(self, x: torch.Tensor) -> bool:
        return (self.stem_packed is not None and self._stem_fused and torch.backends.cudnn.allow_tf32
                and x.dim() == 4 and x.shape[1] == 3 and x.shape[2] % 2 == 0 and x.shape[3] % 2 == 0)

    def stem_forward(self, x: torch.Tensor, normalize=None) -> torch.Tensor:
        """Children 0-3: conv1 + bn1 + relu + maxpool. One fused kernel (gh_stem_conv_pool_nhwc) when the chain below
        would run in TF32 anyway (cudnn.allow_tf32, the torch default) on an fp32 plan; the chain otherwise.
        normalize: (mean, std) for a uint8 batch, ToTensor + Normalize bit for bit as ops.normalize_u8 -- inside the
        fused kernel where it applies (gh_stem_conv_pool_u8_nhwc: no fp32 batch), by normalize_u8 before the chain else."""
        if normalize is not None and x.dtype == torch.uint8:
            if self._fused_stem_applies(x):
                return ops.stem_conv_pool_u8(x, *normalize, self.stem_packed, self.stem_s2d[1])
            x = ops.normalize_u8(x, *normalize)
        if x.dtype == torch.float32 and self._fused_stem_applies(x):
            return ops.stem_conv_pool(x, self.stem_packed, self.stem_s2d[1])
        if (self.stem_s2d is not None and x.dtype == torch.float32 and x.shape[1] == 3 and x.shape[2] % 2 == 0
                and x.shape[3] % 2 == 0):
            x = self._conv_relu(ops.stem_space_to_depth(x, self.dtype), self.stem_s2d)
        else:
            x = x.to(self.dtype)
            if self.channels_last:
                x = x.contiguous(memory_format=torch.channels_last)
            x = self._conv_relu(x, self.stem)
        return self._pool(x)

    def __call__(self, x: torch.Tensor, normalize=None):
        x = self.stem_forward(x, normalize)
        outs = []
        for blocks in self.stages:
            for c1, c2, c3, down in blocks:
                identity = x
                y = self._conv_relu(x, c1)
                y = self._conv_relu(y, c2)
                if down is not None:
                    identity = F.conv2d(x, down[0], down[1], down[2], down[3], down[4], down[5])
                w, b, stride, padding, dilation, groups = c3
                x = torch.cudnn_convolution_add_relu(y, w, identity, 1.0, b, stride, padding, dilation, groups)
            outs.append(x)
        return x, outs
