"""BaseLoss -- the reference's loss-class interface (loss/base_loss.py:9-295) with the
heavy work done by the sm_100a kernels.  Same constructor, attributes, lifecycle hooks and
``compute_base_loss`` signature, so Hydra can instantiate it by changing ``_target_`` only.

What differs under the hood (results are the reference's, SURVEY appendix B):
  * one fused kernel produces CE / weighted CE, the focal term, arg-max, the distill mask
    and d(loss)/d(logits) -- the [B,T,H,W] seen-probability tensor is never materialised;
  * no host synchronisation: "prototypes ready", "batch has background" and the class
    weight normaliser are device-side predicates / scalars."""
from __future__ import annotations

import math
import weakref
from typing import Optional

import numpy as np
import torch

from .. import _cabi, ops
from ..autograd import PixelLossFunction
from ..training.loss_utils import (UnbiasedKnowledgeDistillationLoss, WeightedCrossEntropy)


class FocalSpec:
    """Parameters of the binary seen-detector focal loss (the reference instantiates
    segmentation_models_pytorch.losses.FocalLoss(mode='binary', reduction='mean'),
    base_loss.py:63-70; here the loss is evaluated inside the fused pixel kernel)."""

    def __init__(self, gamma=2.0, alpha=None, ignore_index=255):
        self.gamma, self.alpha, self.ignore_index = float(gamma), alpha, ignore_index


class SeenMap:
    """Stand-in for the reference's ``seen_prob`` [B,T,H,W] tensor: the low-res head
    logits plus what the fused kernel already derived from them."""

    def __init__(self, z: torch.Tensor, distill_mask: Optional[torch.Tensor], scale: int = 16):
        self.z, self.distill_mask, self.scale = z, distill_mask, scale

    def materialize(self) -> torch.Tensor:
        """sigmoid(upsample(z)) exactly as get_seen_probs returns it (bg_detector.py:141-165)."""
        return ops.seen_upsample(self.z, self.scale, apply_sigmoid=True)


class BaseLoss:
    """Parent class for losses (reference: loss/base_loss.py:9)."""

    def __init__(self, name, ignore_index=255):
        self.name = name
        self.old_classes = 0
        self.initial_classes = 0
        self.increment = 0
        self.nb_current_classes = 0
        self.nb_new_classes = 0
        self.epoch_number = 0
        self.max_epochs = 0
        self.device = None
        self.ignore_index = ignore_index
        self._prototypes = None
        self.accelerator = None
        self.seen_fgloss = None
        self.init_seen_focal_loss()
        self.same_task = False
        self.last_task = False
        self.first_task = True
        self.weighted_ce = None
        self.prev_model = None
        self.init_weighted_loss()
        # opt-in, not in the reference: evaluate the network's final logit up-sample inside the loss kernel (see
        # compute_base_loss); False keeps the reference's data flow ([B,K,H,W] logits from the network)
        self.fused_logit_upsample = False
        # opt-in, not in the reference: at world size > 1 keep the exact-mode prototype sums, over the rows of the
        # global batch (Prototypes(exact_across_ranks=True)); False sums per channel there
        self.exact_prototypes_across_ranks = False
        # fused-kernel by-products of the last compute_base_loss call
        self._fused_preds = None
        self._fused_logits_ref = None
        self._fused_distill_mask = None

    # ---- configuration ------------------------------------------------------------------
    def set_device(self, device):
        self.device = device

    def init_seen_focal_loss(self, gamma=2, alpha=None):
        self.seen_fgloss = FocalSpec(gamma=gamma, alpha=alpha, ignore_index=self.ignore_index)

    def init_weighted_loss(self, gamma=2, threshold=0.5, ukd=True):
        self.weighted_ce = WeightedCrossEntropy(ignore_index=self.ignore_index, gamma=gamma, threshold=threshold,
                                                ukd=ukd)
        self.weighted_ce.base_loss = self
        self.lkd_loss = UnbiasedKnowledgeDistillationLoss()

    def _update_task(self, task_num):
        """base_loss.py:80-89"""
        self.nb_new_classes = self.increment
        self.old_classes = self.get_n_old_classes(task_num)
        self.nb_current_classes = self.initial_classes + self.increment * task_num
        self.first_task = task_num == 0

    def get_n_old_classes(self, task_num):
        return self.initial_classes + self.increment * (task_num - 1) if task_num > 0 else 0

    def label_to_task_num(self, label):
        """base_loss.py:98-107: np.rint (half-to-even) of max((label+1-initial)/increment, 0) (Q2)."""
        current_task = 0
        if self.increment > 0:
            if hasattr(label, "cpu"):
                label = label.cpu().numpy()
            current_task = (np.asarray(label) + 1 - self.initial_classes) / self.increment
            current_task[current_task < 0] = 0
            current_task = np.rint(current_task)
        return current_task

    def set_continual_task_size(self, initial_classes, increment=0):
        if self._prototypes is not None:
            self._prototypes.set_continual_task_size(initial_classes, increment)
        self.initial_classes = initial_classes
        self.increment = increment
        self.nb_current_classes = self.initial_classes

    def init_prototype_compute(self):
        from .prototypes import Prototypes
        self._prototypes = Prototypes(name="Prototype_{}".format(self.name), ignore_index=self.ignore_index,
                                      exact_across_ranks=self.exact_prototypes_across_ranks)

    @property
    def prototypes(self):
        return self._prototypes._prototypes_tensors

    def are_prototypes_ready(self):
        """Host bool (synchronises); the hot path uses ``_prototypes.ready_flag`` instead."""
        if self._prototypes is not None:
            return self._prototypes.are_prototypes_ready()
        return False

    # ---- lifecycle events ------------------------------------------------------------------
    def on_fit_start(self, task_num, **kwargs):
        self._update_task(task_num)
        if self._prototypes is not None:
            self._prototypes.on_fit_start(task_num, **kwargs)
            self._prototypes.on_train_start(task_num, **kwargs)

    def on_train_start(self, task_num, **kwargs):
        pass

    def on_train_end(self, **kwargs):
        self._check_cross_rank_state()
        if self._prototypes is not None:
            self._prototypes.on_train_end(**kwargs)

    def on_train_batch_start(self, **kwargs):
        if kwargs.get("batch_idx") == 0 and self.epoch_number is not None and kwargs.get("epoch") != self.epoch_number:
            self._check_cross_rank_state()                 # once per epoch: a cheap host read of one device word
        self.epoch_number = kwargs.get("epoch")
        self.max_epochs = kwargs.get("max_epochs")

    @staticmethod
    def _check_cross_rank_state():
        """Surface a timed-out NVLink prototype exchange (distributed.PeerReducer) as a Python exception at the
        host synchronisation points of the loop (epoch start, end of task).  No-op in single-process runs."""
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            from ..distributed import check_peer_errors
            check_peer_errors()

    # ---- the hot path -------------------------------------------------------------------------
    @staticmethod
    def _heads(seen_fg_network):
        clf = seen_fg_network.seen_not_seen_clf
        return list(clf) if isinstance(clf, torch.nn.ModuleList) else [clf]

    def _stack_heads(self, seen_fg_network, n_heads):
        """[T,D] weights / [T] biases of the heads forward_seen_before evaluates
        (bg_detector.py:119-139): every head of a ModuleList, or the single shared head
        against prototypes[0]."""
        clf = seen_fg_network.seen_not_seen_clf
        heads = list(clf)[:n_heads] if isinstance(clf, torch.nn.ModuleList) else [clf]
        # one cat launch for weights and biases together: [w_0 .. w_{T-1} | b_0 .. b_{T-1}]
        n, d = len(heads), heads[0].conv.weight.numel()
        flat = torch.cat([h.conv.weight.detach().reshape(-1) for h in heads]
                         + [h.conv.bias.detach().reshape(-1) for h in heads]).float()
        return flat[:n * d].view(n, d), flat[n * d:]

    def compute_base_loss(self, img, mask, model, task_num=-1, weights=None, train=True, use_weighted_ce=False,
                          return_attentions=False, _loss_scale=1.0):
        """Reference: base_loss.py:172-253.  Returns ``(loss, logits)`` or, with
        ``return_attentions and train``, ``(loss, logits, old_atts, attentions, seen_map)``
        where ``seen_map`` is a :class:`SeenMap` (call ``.materialize()`` for the tensor)."""
        old_atts, attentions, seen_map = None, None, None
        if self._prototypes is not None and self._prototypes._prototypes_tensors is not None:
            ops.check_task_count(self._prototypes._prototypes_tensors.shape[0], "compute_base_loss")
        is_experience_replay = task_num != -1
        if self.weighted_ce.old_cl != self.old_classes:      # (nn.Module.__setattr__ is slow: only on change)
            self.weighted_ce.old_cl = self.old_classes
        seen_net = getattr(model, "seen_fg_network", None)
        train_seen_detector = (seen_net is not None and (self.same_task or not is_experience_replay) and train)
        return_penultimate = train_seen_detector or use_weighted_ce or self._prototypes is not None
        if self.fused_logit_upsample:
            # opt-in (SURVEY 8f-1): take the head's low-res sem_logits (deeplab_v3.py:155-156) and evaluate the network's
            # final bilinear up-sample (deeplab_v3.py:157-160) and its backward inside the loss kernel
            preds_mask, penultimate_output, attentions = model(img, return_penultimate=True, return_attentions=True,
                                                               return_sem_logits=True)
        else:
            preds_mask, penultimate_output, attentions = model(img, return_penultimate=True, return_attentions=True)
        if self.prev_model is not None and train and return_attentions:
            with torch.no_grad():
                _, _, old_atts = self.prev_model(img, return_penultimate=True, return_attentions=True)
        if return_penultimate and train and self._prototypes is not None:
            self._prototypes.update_feats_prototypes(penultimate_output, mask)
        ready = self._prototypes.ready_flag if self._prototypes is not None else None
        if ready is None:
            train_seen_detector = False
        wce_on = bool(use_weighted_ce and train)
        cfg = {"ignore_index": self.ignore_index, "loss_scale": float(_loss_scale), "want_grad": True,
               "lowres": bool(self.fused_logit_upsample)}
        head_w = head_b = None
        features = penultimate_output
        if wce_on or train_seen_detector:
            protos = self.prototypes
            clf = seen_net.seen_not_seen_clf
            heads = list(clf)[:protos.shape[0]] if isinstance(clf, torch.nn.ModuleList) else [clf]
            params = [h.conv.weight for h in heads] + [h.conv.bias for h in heads]
            if all(p.dtype == torch.float32 and p.is_cuda and p.is_contiguous() for p in params):
                # the kernel reads the heads' own parameters (no gather launch) and clears the focal-gradient
                # accumulator of the pixel kernel that follows (no fill launch)
                n_eval = len(heads)
                if train_seen_detector:
                    cfg["gz"] = torch.empty((penultimate_output.shape[0],) + tuple(penultimate_output.shape[2:]),
                                            dtype=torch.float32, device=penultimate_output.device)
                # more than 32 heads (continual runs longer than 32 tasks): the chunked kernel
                seen = ops.seen_logits_many if n_eval > 32 else ops.seen_logits_heads
                z = seen(penultimate_output.detach(), protos[:n_eval], [p.detach() for p in params[:n_eval]],
                         [p.detach() for p in params[n_eval:]], zero_out=cfg.get("gz"))
            else:
                weight, bias = self._stack_heads(seen_net, protos.shape[0])
                n_eval = weight.shape[0]
                seen = ops.seen_logits_many if n_eval > 32 else ops.seen_logits
                z = seen(penultimate_output.detach(), protos[:n_eval], weight, bias)
            cfg["z"] = z
            cfg["proto"] = protos
        if wce_on:
            if task_num == -1:
                task_num = self.prototypes.shape[0] - 1
            w = self.weighted_ce
            cfg.update(mode=_cabi.PIX_WEIGHTED_CE, old_cl=int(self.old_classes), ukd=bool(w.ukd), gamma=float(w.gamma),
                       threshold=float(w.threshold), want_distill_mask=bool(return_attentions),
                       lkd_threshold=float(getattr(self, "lkd_threshold", 0.5)))
        else:
            # plain / class-weighted CE; without weighted CE the reference has no seen_prob, so the
            # distill mask is (mask == 0) alone (bacs_loss.py:282-285): threshold -1 disables the test
            cfg.update(mode=_cabi.PIX_CE, class_w=weights, want_distill_mask=bool(return_attentions and train),
                       lkd_threshold=-1.0)
        if train_seen_detector:
            head = task_num if (task_num is not None and task_num != -1) else self.prototypes.shape[0] - 1
            heads = self._heads(seen_net)
            head_mod = heads[head] if len(heads) > 1 else heads[0]
            head_w, head_b = head_mod.conv.weight, head_mod.conv.bias
            if hasattr(seen_net, "set_stop_gradients"):
                seen_net.set_stop_gradients(not self.first_task)
            cfg.update(focal_head=int(head), ready=ready, focal_gamma=float(self.seen_fgloss.gamma),
                       focal_alpha=self.seen_fgloss.alpha, features_grad=bool(self.first_task),
                       focal_weight=max(0.0, 1.0 - math.exp(self.epoch_number - self.max_epochs)))
        if not cfg.get("features_grad", False):
            features = penultimate_output.detach()
        if not train:
            cfg["want_grad"] = False
        loss, preds, dmask = PixelLossFunction.apply(preds_mask, features, head_w, head_b, mask, cfg)
        # the arg-max belongs to THIS logits tensor: remember the object itself (weakly) and its version, never id()
        # (CPython reuses the id of a freed tensor, e.g. the replay pass's logits)
        self._fused_preds = preds
        self._fused_logits_ref = (weakref.ref(preds_mask), preds_mask._version, preds_mask.data_ptr())
        dmask = dmask if dmask.numel() else None
        self._fused_distill_mask = dmask
        if wce_on:
            seen_map = SeenMap(cfg["z"], dmask)
        if return_attentions and train:
            return loss, preds_mask, old_atts, attentions, seen_map
        return loss, preds_mask

    def _argmax(self, preds_mask):
        """arg-max of the logits; free when the fused kernel already produced it (bacs_loss.py:255)."""
        ref = getattr(self, "_fused_logits_ref", None)
        if (self._fused_preds is not None and ref is not None and ref[0]() is preds_mask
                and ref[1] == preds_mask._version and ref[2] == preds_mask.data_ptr()):
            return self._fused_preds
        out = ops.pixel_loss(preds_mask.detach(), torch.zeros(preds_mask.shape[0], *preds_mask.shape[2:],
                                                              dtype=torch.int64, device=preds_mask.device),
                             _cabi.PIX_CE, want_grad=False)
        return out["preds"]

    def preprocess_batch(self, batch):
        """base_loss.py:274-282 -- including the .long() of the replay logits (Q4)."""
        if isinstance(batch, dict):
            for key in batch:
                batch[key][0] = batch[key][0].float()
                batch[key][1] = batch[key][1].long()
        else:
            batch[0] = batch[0].float()
            batch[1] = batch[1].long()
        return batch

    def compute_loss(self, batch, model, train=True):
        pass
