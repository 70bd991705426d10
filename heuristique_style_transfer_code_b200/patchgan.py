"""Multi-PatchGAN discriminators with the Gram head on the B200 kernels (SURVEY 8(f) n4).

Drop-in for the two inference classes of the reference's Models/Models_Multi_PatchGAN.py that carry a Gram head
(`VariablePatchesNLayerDiscriminator_test` :113-264 and `MultiScaleDiscriminator_test` :266-322, the ones
test_Multi_PatchGAN.py:11,79 builds): same constructor arguments, same submodules created in the same order (identical
random init under one seed, identical state_dict keys), same `(embeddings, output)` return and `get_gram_norms()`.

What runs where:
  * the convolutional feature extractor and the 1x1 projection convolutions stay on cuDNN (the backbone, as for the
    ResNet model);
  * everything from the collected projections on -- layer norm :198, 4x4 adaptive pooling :210, layer norm :213, the
    D x D Gram over 16 positions :217-220, its Frobenius norm :223, Linear(D*D -> ndf) :229, the two 8-head attentions
    :243-244, the mean over layers :247 and the classifier :256 -- is three launches of the C-ABI library
    (gh_patch_gram_fwd, gh_gemm_f32, gh_patch_attn_fwd). There is no CPU path.

NaN handling. The reference tests every activation with `torch.isnan(x).any()` (:186, :192, :232 -- one host
synchronisation and one extra pass per layer) and, where a NaN is found, prints a message and applies
`torch.nan_to_num(.., nan=0.0)`. A NaN anywhere reaches the embeddings of its image (convolutions, the whole-map layer
norm and the softmax over layers all propagate it), so here the forward runs once without the checks, tests only the
(B, ndf) / (B, nc) results, and -- only if they hold a NaN -- runs again layer by layer with the reference's checks,
messages and replacements. Clean inputs pay one tiny check instead of ~20 synchronisations.

Gradients. By default the kernels serve forwards without autograd history: the classification / evaluation / camera
call sites (functions_Multi_PatchGAN.py:164, :200, :464) run under torch.no_grad(). A forward that needs autograd history
(fine-tuning the discriminator, a GAN loss through it, a regulariser on get_gram_norms(), or `style_transfer_patches`,
functions_Multi_PatchGAN.py:272-287, which optimises an image through it) is handed to the reference's OWN forward
(Models/Models_Multi_PatchGAN.py:177-256, executed on this module's parameters; loaded by _reference.py); when no copy of
the reference is available it raises GramHeadError rather than returning tensors without history.
`set_library_backward(True)` (or GRAMHEAD_PATCHGAN_BACKWARD=1 in the environment, for unmodified scripts) runs such a
forward on the kernels instead, under three autograd Functions that mirror the three launches (ops._PatchGram,
ops._PatchProjection, ops._PatchAttention) and backpropagate on the library's backward kernels. It is opt-in only so
that the default does not move; the next step is to make it the default and delete _reference_forward (DESIGN.md
section 8).
"""
from __future__ import annotations

import functools
import os

import torch
import torch.nn as nn

from . import ops
from ._lib import GramHeadError

PATCH_TYPES = {'small': (4, 30), 'medium': (31, 80), 'large': (81, 150)}          # Models_Multi_PatchGAN.py:11-15


def _library_backward_from_env() -> bool:
    return os.environ.get("GRAMHEAD_PATCHGAN_BACKWARD", "").strip() == "1"


class VariablePatchesNLayerDiscriminator_test(nn.Module):
    def __init__(self, input_nc=3, ndf=64, norm="instance", tensorboard_logdir=None, global_step=None,
                 patch_size=70, num_classes=10, gram_matrix_dim=64, pooling_type='avg'):
        super().__init__()
        self.tensorboard_logdir = tensorboard_logdir
        self.writer = None
        self.global_step = global_step
        self.num_classes = num_classes
        self.gram_matrix_dim = gram_matrix_dim
        self.pooling_type = pooling_type
        self.gram_norms = []

        make_norm = (functools.partial(nn.InstanceNorm2d, affine=False) if norm == 'instance'
                     else functools.partial(nn.BatchNorm2d, affine=True))
        # :129-157  stride-2 4x4 convolutions while the receptive field allows and the width is <= 512, then two
        # stride-1 convolutions; the module names are the state_dict keys
        self.feature_extractor = nn.Sequential()
        width, channels, field, i = ndf, input_nc, patch_size, 0
        while field > 4 and width <= 512:
            self.feature_extractor.add_module(f'conv{i}', nn.Conv2d(channels, width, 4, 2, 1))
            self.feature_extractor.add_module(f'norm{i}', make_norm(width))
            self.feature_extractor.add_module(f'relu{i}', nn.ReLU(inplace=True))
            channels, width, field, i = width, width * 2, field / 2, i + 1
        self.feature_extractor.add_module('final_conv', nn.Conv2d(channels, width, 4, 1, 1))
        self.feature_extractor.add_module('final_norm', make_norm(width))
        self.feature_extractor.add_module('final_relu', nn.ReLU(inplace=True))
        self.feature_extractor.add_module('final_conv_ndf', nn.Conv2d(width, ndf, 4, 1, 1))

        # :160-165  one 1x1 projection to gram_matrix_dim channels per convolution, in module order
        self.projection_layers = nn.ModuleList(
            nn.Conv2d(m.out_channels, gram_matrix_dim, kernel_size=1)
            for m in self.feature_extractor if isinstance(m, nn.Conv2d))
        self.attention_per_layer = nn.MultiheadAttention(embed_dim=ndf, num_heads=8)       # :168-169
        self.attention_per_patch = nn.MultiheadAttention(embed_dim=ndf, num_heads=8)
        self.classifier = nn.Linear(ndf, num_classes)                                      # :172
        self.feature_projection = nn.Linear(gram_matrix_dim * gram_matrix_dim, ndf)        # :175
        # plain attribute (no state_dict key): grad-enabled forwards on the library's kernels instead of the reference's
        self.library_backward = _library_backward_from_env()

    def set_library_backward(self, enabled: bool = True):
        """Run forwards that need autograd history on the library's kernels and backward kernels (see the module
        docstring). Returns self."""
        self.library_backward = bool(enabled)
        return self

    # -- the head ------------------------------------------------------------------------------------------------------
    def _needs_autograd(self, x):
        return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))

    def _reference_forward(self, x):
        """The reference's own forward on this module's parameters (differentiable; see the module docstring)."""
        from ._reference import load_reference_file
        try:
            ref = load_reference_file(os.path.join("Models", "Models_Multi_PatchGAN.py"))
        except NotImplementedError as exc:
            raise GramHeadError("gramhead: the Multi-PatchGAN Gram head kernels are inference-only and no copy of the "
                                "reference is available for a forward that needs gradients: call the model under "
                                "torch.no_grad(), or " + str(exc)) from exc
        return ref.VariablePatchesNLayerDiscriminator_test.forward(self, x)

    def _forward(self, x, careful: bool, grad: bool = False):
        maps, k = [], 0
        for idx, layer in enumerate(self.feature_extractor):
            x = layer(x)
            if careful and torch.isnan(x).any():
                print(f"NaN detected after layer {idx}")
                x = torch.nan_to_num(x, nan=0.0)
            if isinstance(layer, nn.Conv2d):
                x_proj = self.projection_layers[k](x)
                if careful and torch.isnan(x_proj).any():
                    print(f"NaN detected in projected feature map at layer {idx}")
                    x_proj = torch.nan_to_num(x_proj, nan=0.0)
                maps.append(x_proj.float())
                k += 1
        if not maps:
            raise ValueError("No feature maps were collected. Check the model architecture and input data.")
        # layer norm :198 is folded into the pooling pass (pooling is linear, the norm a per-image affine map)
        if grad:
            gram, norms = ops.patch_gram_autograd(maps, ln_input=True)
            feat = ops.patch_projection_autograd(gram, self.feature_projection)
        else:
            gram, norms = ops.patch_gram(maps, ln_input=True)
            L, b, dd = gram.shape
            feat = ops.gemm_f32(gram.view(L * b, dd), self.feature_projection.weight.detach().t(),
                                self.feature_projection.bias.detach()).view(L, b, -1)
        if careful:
            bad = torch.isnan(feat).flatten(1).any(dim=1).tolist()
            rows = list(feat.unbind(0)) if grad else None      # out of place under autograd: nan_to_num's own gradient
            for fm_idx, flag in enumerate(bad):
                if flag:
                    print(f"NaN detected in projected features at layer {fm_idx}, replacing NaNs with zeros.")
                    if grad:
                        rows[fm_idx] = torch.nan_to_num(rows[fm_idx], nan=0.0)
                    else:
                        feat[fm_idx] = torch.nan_to_num(feat[fm_idx], nan=0.0)
            if grad:
                feat = torch.stack(rows, dim=0)
        if grad:
            emb, out = ops.patch_attention_autograd(feat, self.attention_per_layer, self.attention_per_patch,
                                                    self.classifier)
        else:
            emb, out = ops.patch_attention(feat, self.attention_per_layer, self.attention_per_patch, self.classifier)
        return emb, out, norms

    def forward(self, input):
        assert input.ndim == 4, f"Input must be NCHW, got {input.shape}"
        if not input.is_cuda:
            raise GramHeadError(f"gramhead: input must be a CUDA tensor (got {input.device}); the head has no CPU path")
        if self._needs_autograd(input):
            if not self.library_backward:
                return self._reference_forward(input)
            emb, out, norms = self._forward(input, careful=False, grad=True)
            if bool(torch.isnan(emb).any() | torch.isnan(out).any()):
                emb, out, norms = self._forward(input, careful=True, grad=True)
            self.gram_norms = list(norms.unbind(0))
            return emb, out
        with torch.no_grad():
            emb, out, norms = self._forward(input, careful=False)
            if bool(torch.isnan(emb).any() | torch.isnan(out).any()):
                emb, out, norms = self._forward(input, careful=True)
        self.gram_norms = list(norms.unbind(0))
        return emb, out

    def get_gram_norms(self):
        return self.gram_norms


class MultiScaleDiscriminator_test(nn.Module):
    def __init__(self, input_nc=3, ndf=64, norm='batch', tensorboard_logdir=None, global_step=None,
                 patch_sizes={'small': 10, 'medium': 70, 'large': 150}, num_classes=10,
                 gram_matrix_dim=64, pooling_type='avg'):
        super().__init__()
        self.patch_sizes = patch_sizes
        self.tensorboard_logdir = tensorboard_logdir
        self.global_step = global_step
        self.scale_discriminators = nn.ModuleDict()
        for patch_type in PATCH_TYPES:                               # :283-299: every scale sees the same input
            logdir = os.path.join(tensorboard_logdir, patch_type) if tensorboard_logdir else None
            self.scale_discriminators[patch_type] = VariablePatchesNLayerDiscriminator_test(
                input_nc=input_nc, patch_size=patch_sizes.get(patch_type, 70), ndf=ndf, norm=norm,
                tensorboard_logdir=logdir, global_step=global_step, num_classes=num_classes,
                gram_matrix_dim=gram_matrix_dim, pooling_type=pooling_type)

    def set_library_backward(self, enabled: bool = True):
        """set_library_backward of every scale. Returns self."""
        for discriminator in self.scale_discriminators.values():
            discriminator.set_library_backward(enabled)
        return self

    def forward(self, input):
        embs, outs = [], []
        for discriminator in self.scale_discriminators.values():
            e, o = discriminator(input)
            embs.append(e)
            outs.append(o)
        return torch.stack(embs, dim=0).mean(dim=0), torch.stack(outs, dim=0).mean(dim=0)     # :309-311

    def get_gram_norms(self):
        norms = []
        for discriminator in self.scale_discriminators.values():
            norms.extend(discriminator.get_gram_norms())
        return norms


# ----------------------------------------------------------------------------------------------------------------------
# The training-time classes of the same file (:17-110) have no Gram head (plain convolution stacks on cuDNN) and are
# outside this package's path: `VariablePatchesNLayerDiscriminator` / `MultiScaleDiscriminator` resolve lazily to the
# reference's own classes (train_best_Multi_PatchGAN.py:11 imports MultiScaleDiscriminator from this module path).
# ----------------------------------------------------------------------------------------------------------------------
_REFERENCE_ONLY = ("VariablePatchesNLayerDiscriminator", "MultiScaleDiscriminator")


def __getattr__(name):
    if name in _REFERENCE_ONLY:
        from ._reference import load_reference_file
        return getattr(load_reference_file(os.path.join("Models", "Models_Multi_PatchGAN.py")), name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
