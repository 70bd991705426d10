"""Drop-in nn.Modules for the reference's Gram + attention classifier.

Mirrors Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py (reference tree): class names, constructor signature
(:14 / :66), public attributes (device, truncated_encoder, num_classes, gram_matrix_size, classifier, attention),
gram_matrix() (:26-30), forward() return conventions (:61 logits | :113-114 (embeddings, logits)), the zero-stage early
return (:48-49) and therefore the state_dict keys (truncated_encoder.*, classifier.{weight,bias},
attention.{in_proj_weight,in_proj_bias,out_proj.weight,out_proj.bias}). Submodules are created in the reference's order
(encoder, classifier, attention) so a seeded construction consumes the RNG identically.

What differs is how forward() computes: the backbone stays on cuDNN (as the task prescribes), everything after it --
Gram, pooling, token layout, attention, mean, classifier and their backward -- runs in libgramhead.so's sm_100a
kernels (ops.py). nn.MultiheadAttention / nn.Linear are kept purely as parameter containers. The module does not turn
on torch.autograd.set_detect_anomaly (the reference does so at import, :9).
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from . import ops
from .frozen_encoder import FoldedEncoder, encoder_signature

# How the cuDNN backbone hands its stage activations to the head (SURVEY.md section 8(f) n1):
#   "reference"          - exactly the reference's execution: fp32 NCHW, torch defaults (the default on CPU)
#   "channels_last"      - fp32 as above, encoder and activations in channels_last (NHWC): same precision and the same
#                          cuDNN convolutions, minus cuDNN's internal NCHW<->NHWC conversion kernels (12 % of the encoder
#                          in the reference mode) and with the NHWC batch-norm kernels: logits differ by 1e-7 from the
#                          reference mode, the training step is 1.6x faster (85 -> 53 ms at batch 256). Default on CUDA.
#   "bf16"               - torch.autocast(bfloat16) around the encoder: bf16 NCHW activations
#   "bf16_channels_last" - encoder converted to channels_last and run under bf16 autocast: bf16 NHWC activations
# The bf16 modes change the numerics of the BACKBONE (not of the head) and are opt-in: model.set_backbone_mode(...) or
# the environment variable GRAMHEAD_BACKBONE for unmodified reference scripts (GRAMHEAD_BACKBONE=reference restores
# the NCHW execution).
BACKBONE_MODES = ("reference", "channels_last", "bf16", "bf16_channels_last")
# Inference plan (frozen_encoder.py): in the two channels_last modes, with the module in eval mode and gradients disabled,
# eval-mode batch norm is folded into the convolution before it and ReLU / residual add run as cuDNN epilogues -- the
# same function, the same cuDNN convolutions, without the element-wise passes that are 69 % of the encoder's time.
# model.fold_batchnorm = False (or GRAMHEAD_FOLD_BN=0) executes the children one by one as the reference does.


class GramAttentionHead:
    """Functional core shared by both classes: stage activations -> (embeddings, logits)."""

    @staticmethod
    def apply(stages, gram_matrix_size: int, attention: nn.MultiheadAttention, classifier: nn.Linear):
        desc = ops.style_descriptor(stages, gram_matrix_size)
        return ops.attention_head(desc, attention.in_proj_weight, attention.in_proj_bias, attention.out_proj.weight,
                                  attention.out_proj.bias, classifier.weight, classifier.bias)


class _TruncatedGramAttentionBase(nn.Module):
    def __init__(self, base_encoder, truncate_after_layer, num_classes, gram_matrix_size, device='cpu'):
        super().__init__()
        self.device = device
        self.truncated_encoder = nn.Sequential(*list(base_encoder.children())[:truncate_after_layer]).to(self.device)
        self.num_classes = num_classes
        self.gram_matrix_size = gram_matrix_size
        self.classifier = nn.Linear(self.gram_matrix_size ** 2, self.num_classes).to(self.device)
        self.attention = nn.MultiheadAttention(embed_dim=self.gram_matrix_size ** 2, num_heads=1).to(self.device)
        self._backbone_mode = "reference"
        self.fold_batchnorm = os.environ.get("GRAMHEAD_FOLD_BN", "1") != "0"
        self._plan = None
        self._input_normalization = None
        on_cuda = torch.device(self.device).type == "cuda"
        env_mode = os.environ.get("GRAMHEAD_BACKBONE", "")
        if env_mode or on_cuda:
            self.set_backbone_mode(env_mode or "channels_last")

    @property
    def backbone_mode(self) -> str:
        return self._backbone_mode

    def set_backbone_mode(self, mode: str):
        """Selects how the encoder runs (see BACKBONE_MODES). Parameters, state_dict keys and dtypes are unchanged."""
        if mode not in BACKBONE_MODES:
            raise ValueError(f"backbone mode must be one of {BACKBONE_MODES}, got {mode!r}")
        fmt = torch.channels_last if mode.endswith("channels_last") else torch.contiguous_format
        self.truncated_encoder.to(memory_format=fmt)
        self._backbone_mode = mode
        return self

    @property
    def input_normalization(self):
        """((mean, mean, mean), (std, std, std)) applied to (B, 3, H, W) uint8 input, or None (the default)."""
        return self._input_normalization

    def set_input_normalization(self, mean, std=None):
        """Lets forward() take the uint8 pixels of the loaders (functions.uint8_transform): a (B, 3, H, W) uint8 batch is
        then transformed by ToTensor + Normalize(mean, std) first, bit for bit as ops.normalize_u8 / the host transforms
        (reference test_...:64-65), so model(x_u8) == model(normalized x_u8). On the fp32 inference plan with the fused
        stem this happens inside the stem kernel and no fp32 batch is built. Other input is unaffected.
        set_input_normalization(None) turns it off. A plain attribute: no buffer, no state_dict key. Returns self."""
        if mean is None:
            if std is not None:
                raise ValueError("set_input_normalization(None) takes no std")
            self._input_normalization = None
            return self
        mean, std = tuple(float(v) for v in mean), tuple(float(v) for v in std)
        if len(mean) != 3 or len(std) != 3:
            raise ValueError(f"input normalisation needs 3 means and 3 stds, got {len(mean)} and {len(std)}")
        if not all(s != 0.0 and s == s for s in std):
            raise ValueError(f"input normalisation: std must be non-zero, got {std}")
        self._input_normalization = (mean, std)
        return self

    def gram_matrix(self, activations):
        """(b, ch, h, w) -> (b, ch, ch): F F^T / (h*w), differentiable (dense tcgen05 Gram kernels)."""
        return ops.gram_matrix(activations)

    def train(self, mode: bool = True):
        # Weights are about to change (train) or have just changed (eval after training): the folded encoder copies and the
        # cached split planes of the attention weights are rebuilt at the next inference forward. Version counters alone
        # cannot be trusted for this -- fused optimizers update parameters without bumping them.
        # A call that changes nothing (eval() on a model already in eval mode) keeps them: captured CUDA graphs
        # (streaming.CameraPipeline) hold the addresses of the folded tensors.
        if mode or self.training != mode:
            self._plan = None
            ops.clear_weight_planes()
        return super().train(mode)

    def refresh_inference_plan(self):
        """Drops the folded weight copies. Only needed after editing encoder tensors through `.data` (which bypasses
        the version counters the plan watches); optimizer steps, load_state_dict, .to() and train() are detected."""
        self._plan = None
        return self

    def _inference_plan(self, x):
        """The folded encoder when it computes the same function as the children (see frozen_encoder.py), else None."""
        if torch.is_grad_enabled():
            if self._plan is not None and any(p.requires_grad for p in self.truncated_encoder.parameters()):
                self._plan = None          # a gradient-enabled forward over trainable weights: an update may follow
            return None
        if not (self.fold_batchnorm and self._backbone_mode.endswith("channels_last")):
            return None
        enc = self.truncated_encoder
        if not x.is_cuda or any(m.training for m in enc.modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)):
            return None
        dtype = torch.bfloat16 if self._backbone_mode.startswith("bf16") else torch.float32
        plan = self._plan
        signature = encoder_signature(enc)
        if signature is None:
            return None
        if plan is None or plan.dtype != dtype or plan.signature != signature:
            plan = FoldedEncoder.build(enc, dtype, channels_last=True) if FoldedEncoder.supported(enc) else None
            self._plan = plan
        return plan

    def _stage_activations(self, x, *, normalize=None):
        """normalize: (mean, std) to use in place of input_normalization for this call (streaming.FrameBatchPipeline
        feeds uint8 batches without changing the model)."""
        x = x.to(self.device)
        norm = self._input_normalization if normalize is None else normalize
        if norm is not None and not (x.dtype == torch.uint8 and x.dim() == 4 and x.shape[1] == 3):
            norm = None
        plan = self._inference_plan(x)
        if plan is not None:
            return plan(x, normalize=norm)
        if norm is not None:
            x = ops.normalize_u8(x, *norm) if x.is_cuda else ops.normalize_u8_host(x, *norm)
        if self._backbone_mode == "reference":
            return self._run_encoder(x)
        if self._backbone_mode.endswith("channels_last"):
            x = x.contiguous(memory_format=torch.channels_last)
        if self._backbone_mode == "channels_last":
            return self._run_encoder(x)
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
            return self._run_encoder(x)

    def _run_encoder(self, x):
        enc = self.truncated_encoder
        # conv1, bn1, relu, maxpool -- an encoder truncated below 4 children raises IndexError, as the reference does
        x = enc[0](x)
        x = enc[1](x)
        x = enc[2](x)
        x = enc[3](x)
        stages = []
        for block in enc[4:]:
            x = block(x)
            stages.append(x)
        return x, stages

    def _head(self, x, *, normalize=None):
        x, stages = self._stage_activations(x, normalize=normalize)
        if not stages:
            return None, torch.zeros((x.size(0), self.num_classes), requires_grad=True).to(self.device)
        return GramAttentionHead.apply(stages, self.gram_matrix_size, self.attention, self.classifier)


class TruncatedResNet50(_TruncatedGramAttentionBase):
    """Training variant: forward(x) -> logits (B, num_classes)."""

    def forward(self, x):
        _, logits = self._head(x)
        return logits


class TruncatedResNet50_for_test(_TruncatedGramAttentionBase):
    """Evaluation variant: forward(x) -> (embeddings (B, g*g), logits (B, num_classes)).
    With no Gram stages it returns the zero logits alone, exactly like the reference (:100-101)."""

    def forward(self, x):
        emb, logits = self._head(x)
        if emb is None:
            return logits
        return emb, logits
