"""BgDetector -- drop-in for the reference's ``networks.bg_detector`` (networks/bg_detector.py).

``base_layers`` (conv3x3 + BN + ReLU + Dropout) is network-side and stays on cuDNN; the
per-task heads -- sigmoid/L1 distance to the task prototype, 1x1 conv, x16 bilinear
up-sample -- run on the seen-logits kernels (csrc/seen.cu).  The head modules keep the
reference's parameter layout (``conv.weight`` [1,D,1,1], ``conv.bias`` [1]) so state dicts
are interchangeable."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops


class _SeenLogitsFunction(torch.autograd.Function):
    """z = bias + sum_c w_c |sigmoid(x_c) - sigmoid(p_c)| for one head, at feature resolution."""

    @staticmethod
    def forward(ctx, x, prototype, weight, bias, stop_gradients: bool):
        z = ops.seen_logits(x.detach(), prototype.detach().reshape(1, -1), weight.detach().reshape(1, -1),
                            bias.detach().reshape(1))
        ctx.save_for_backward(x, prototype, weight)
        ctx.stop = stop_gradients
        ctx.shapes = (weight.shape, bias.shape)
        return z

    @staticmethod
    def backward(ctx, gz):
        x, prototype, weight = ctx.saved_tensors
        want_dx = ctx.needs_input_grad[0] and not ctx.stop
        dw, db, dx = ops.seen_head_backward(x.detach(), prototype.detach().reshape(-1).float().contiguous(),
                                            weight.detach().reshape(-1).float().contiguous(),
                                            gz[:, 0].float().contiguous(), None, want_dx)
        return dx, None, dw.reshape(ctx.shapes[0]).to(weight.dtype), db.reshape(ctx.shapes[1]).to(weight.dtype), None


class classification_head(nn.Module):
    def __init__(self, feat_dim, num_classes, stop_gradients=False) -> None:
        super().__init__()
        if num_classes != 1:
            raise NotImplementedError("classification_head: the reference only ever builds 1-output heads "
                                      "(learner/baselearner.py:18-24)")
        self.feat_dim = feat_dim
        self.conv = nn.Conv2d(self.feat_dim, num_classes, 1)
        self.norm = nn.Sigmoid()
        self.stop_gradients = stop_gradients
        self.upsampling_layer = nn.Sequential(nn.Upsample(scale_factor=16, mode="bilinear", align_corners=True))

    def get_distance(self, x, prototype):
        """|sigmoid(x) - sigmoid(prototype)| (bg_detector.py:17-33); plain tensor ops, for inspection."""
        if self.stop_gradients:
            x, prototype = x.detach(), prototype.detach()
        return torch.abs(self.norm(x) - self.norm(prototype))

    def predict_lowres(self, x, prototype):
        return _SeenLogitsFunction.apply(x, prototype.reshape(-1), self.conv.weight, self.conv.bias,
                                         bool(self.stop_gradients))

    def predict(self, x, prototype):
        """bg_detector.py:35-40.  The low-res logits come from the CUDA kernel; with autograd
        off the x16 up-sample does too, otherwise torch's interpolate carries the gradient."""
        z = self.predict_lowres(x, prototype)
        if not torch.is_grad_enabled() or not z.requires_grad:
            return ops.seen_upsample(z, 16, apply_sigmoid=False)
        return self.upsampling_layer(z)

    def forward(self, prototype, x):
        return self.predict(x, prototype)


class BgDetector(nn.Module):
    def __init__(self, in_channels: int) -> None:
        super().__init__()
        self.stop_gradients = False
        self.inter_channels = in_channels // 4
        self.base_layers = nn.Sequential(
            nn.Conv2d(in_channels, self.inter_channels, 3, padding=1, bias=False),
            nn.BatchNorm2d(self.inter_channels), nn.ReLU(), nn.Dropout(0.1))
        self.seen_not_seen_clf = None

    def set_stop_gradients(self, stop_grads):
        if self.seen_not_seen_clf is None or stop_grads == self.stop_gradients:
            return
        self.stop_gradients = stop_grads
        heads = self.seen_not_seen_clf if isinstance(self.seen_not_seen_clf, nn.ModuleList) else [self.seen_not_seen_clf]
        for layer in heads:
            layer.stop_gradients = stop_grads

    def get_classification_head(self, num_classes):
        return classification_head(self.inter_channels, num_classes, stop_gradients=self.stop_gradients)

    def get_penultimate_output(self, x):
        return self.base_layers(x)

    def get_penultimate_layer_dim(self):
        return self.inter_channels

    def get_seen_map_task(self, penultimate_output, prototype, task_num):
        """bg_detector.py:100-117: free logits [B,1,H,W] of one task head."""
        clf = self.seen_not_seen_clf
        head = clf[task_num] if isinstance(clf, nn.ModuleList) else clf
        return head.predict(penultimate_output, prototype[task_num])

    def _stacked(self, n_heads):
        clf = self.seen_not_seen_clf
        heads = list(clf)[:n_heads] if isinstance(clf, nn.ModuleList) else [clf]
        w = torch.cat([h.conv.weight.detach().reshape(1, -1) for h in heads], 0)
        b = torch.cat([h.conv.bias.detach().reshape(1) for h in heads], 0)
        return w, b

    def forward_seen_before_lowres(self, x, prototypes):
        """All heads at feature resolution in one kernel (no gradient): [B,T,h,w]."""
        w, b = self._stacked(prototypes.shape[0])
        seen = ops.seen_logits_many if w.shape[0] > 32 else ops.seen_logits
        return seen(x.detach(), prototypes[:w.shape[0]].detach(), w, b)

    def forward_seen_before(self, x, prototypes):
        """bg_detector.py:119-139 (no gradient -- the loss only uses it under no_grad)."""
        return ops.seen_upsample(self.forward_seen_before_lowres(x, prototypes), 16, apply_sigmoid=False)

    def get_seen_probs(self, x, prototypes, bg_detect=False):
        """bg_detector.py:141-165: sigmoid of every head's up-sampled logits, [B,T,H,W]."""
        return ops.seen_upsample(self.forward_seen_before_lowres(x, prototypes), 16, apply_sigmoid=True)
