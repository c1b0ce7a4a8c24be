"""Prototypes -- per-task running-mean feature prototypes (reference: loss/prototypes.py).

The label-masked feature sums are a segmented reduction on the GPU
(csrc/labels.cu + csrc/prototypes.cu); the "is ready" predicate and the "no foreground in
this batch" early-out are device-side, so ``update_feats_prototypes`` never synchronises.

``exact=True`` (default) reproduces the reference bit-for-bit in structure, including the
channel-scrambled row sums of ``features[mask.expand(..)].view(D, -1)`` for B > 1 (Q1).
``exact=False`` is the per-channel sum the reference computes for B == 1.

Across data-parallel ranks (``sync_across_ranks`` with world size > 1) the sums of the ranks
are added up.  By default the exact mode is dropped there for the per-channel sum (the sums
then equal those of a single process fed every rank's images one by one).
``exact_across_ranks=True`` keeps it: one extra exchange of every rank's per-task pixel
counts gives each rank its images' rows in the view of the global batch, so prototypes and
counts equal those of one process fed the concatenation of the ranks' batches in rank order.
It costs one more cross-rank wait per step, before the sums.  At world size 1 it has no
effect."""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .. import ops
from .base_loss import BaseLoss


class Prototypes(BaseLoss):
    def __init__(self, name="Prototypes", ignore_index=255, exact: bool = True, sync_across_ranks: bool = True,
                 exact_across_ranks: bool = False):
        super().__init__(name, ignore_index)
        self._prototypes_tensors = None
        self._count_features = None
        self.exact = exact
        self.sync_across_ranks = sync_across_ranks
        self.exact_across_ranks = exact_across_ranks
        self.ready_flag: Optional[torch.Tensor] = None     # int32 [1] on the device
        self._task_lut = None
        self._task_lut_key = None

    @property
    def prototypes(self):
        return self._prototypes_tensors

    # ---- ready predicate ---------------------------------------------------------------------
    def refresh_ready(self):
        """Recomputes the device flag from the counts (needed only after the counts were
        assigned from outside, e.g. on resume)."""
        if self._count_features is None:
            self.ready_flag = None
        else:
            self.ready_flag = (self._count_features != 0).all().to(torch.int32).reshape(1)
        return self.ready_flag

    def are_prototypes_ready(self):
        """prototypes.py:31-40 (host bool; synchronises -- not used on the hot path)."""
        return (self._count_features is not None
                and int(self._count_features.count_nonzero()) == self._count_features.shape[0])

    # ---- lifecycle ---------------------------------------------------------------------------
    def on_train_start(self, task_num, **kwargs):
        model = kwargs.get("model")
        accelerator = kwargs.get("accelerator")
        self._init_prototypes(task_num, accelerator, model.get_penultimate_layer_dim())

    def _init_prototypes(self, task_num, accelerator, penultimate_dim):
        """prototypes.py:53-90: one more zero row per task; counts are int64 on the first
        task and become float32 through the first torch.cat with float zeros (Q3)."""
        device = accelerator.root_device
        if task_num > 0:
            self._prototypes_tensors = torch.cat(
                [self._prototypes_tensors, torch.zeros([1, penultimate_dim], device=device)], dim=0)
            self._count_features = torch.cat([self._count_features, torch.zeros([1], device=device)], dim=0)
        else:
            self._prototypes_tensors = torch.zeros([1, penultimate_dim], device=device)
            self._count_features = torch.zeros([1], dtype=torch.long, device=device)
        self._prototypes_tensors.requires_grad = False
        self._count_features.requires_grad = False
        self.refresh_ready()

    def on_train_end(self, **kwargs):
        """prototypes.py:92-125: back-fill prototypes over the train loader when some task
        still has no sample (the recompute-on-resume path)."""
        model = kwargs.get("model", None)
        train_dataloader = kwargs.get("train_dataloader", None)
        accelerator = kwargs.get("accelerator", None)
        if model is None or train_dataloader is None or accelerator is None:
            return
        if not self.are_prototypes_ready():
            append_media = kwargs.get("log_media")
            model = model.to(accelerator.root_device)
            train_dataloader = accelerator.process_dataloader(train_dataloader)
            for batch in train_dataloader:
                batch = accelerator.to_device(batch)
                images, labels = batch[0], batch[1]
                labels = labels.long()
                self.update_prototypes(model, images, labels)
                if append_media is not None:
                    append_media({"inputs": images, "labels": labels})

    # ---- the update --------------------------------------------------------------------------
    def _device_task_lut(self, device, n_tasks):
        key = (self.initial_classes, self.increment, self.ignore_index, n_tasks, str(device))
        if self._task_lut_key != key:
            lut = np.asarray(self.label_to_task_num(np.arange(256, dtype=np.int64)), dtype=np.float64)
            lut = np.broadcast_to(lut, (256,)).astype(np.int64).copy()
            lut[0] = -1                                   # background never owns a prototype (include_bg=False)
            if 0 <= self.ignore_index < 256:
                lut[self.ignore_index] = -1
            lut[lut >= n_tasks] = -1                      # classes of tasks not created yet
            self._task_lut = torch.from_numpy(lut.astype(np.int32)).to(device)
            self._task_lut_key = key
        return self._task_lut

    def update_feats_prototypes(self, features, target, labels_down=None):
        """prototypes.py:127-163.  features [B,D,h,w] (any of fp32/bf16/fp16), target
        [B,H,W] int64; optional labels_down [B,1,h,w] as in the reference."""
        if self._prototypes_tensors is None:
            raise RuntimeError("Prototypes: _init_prototypes has not run (on_fit_start / on_train_start)")
        features = features.detach()
        B, D, h, w = features.shape
        T = self._prototypes_tensors.shape[0]
        labels = target if labels_down is None else labels_down.reshape(B, h, w)
        if labels.dtype != torch.int64:
            labels = labels.long()
        lut = self._device_task_lut(features.device, T)
        task, rank, n_bt, _ = ops.label_downsample_task(labels, h, w, lut, T)
        world = 1
        if self.sync_across_ranks and torch.distributed.is_available() and torch.distributed.is_initialized():
            world = torch.distributed.get_world_size()
        global_view = self.exact and self.exact_across_ranks and world > 1
        mode = 0 if (self.exact and world == 1) or global_view else 1
        if not self._prototypes_tensors.is_contiguous():
            self._prototypes_tensors = self._prototypes_tensors.contiguous()
        if world > 1:
            from ..distributed import allreduce_packed, exchange_task_counts, peer_reducer
            packed = torch.empty(T * D + T, dtype=torch.float64, device=features.device)
            if global_view:
                reducer = peer_reducer(packed.numel(), features.device)
                view_pre, view_n = exchange_task_counts(n_bt, reducer)
                sums, counts = ops.proto_accumulate_view(features, task, rank, n_bt, T, view_pre, view_n, out=packed)
            else:
                sums, counts = ops.proto_accumulate(features, task, rank, n_bt, T, mode, out=packed)
                reducer = peer_reducer(packed.numel(), features.device)
            if reducer is not None and self._count_features.is_contiguous():
                # one launch: sum over the ranks through NVLink peer memory + running-mean update
                self.ready_flag = reducer.allreduce(packed, self._prototypes_tensors, self._count_features, T, D)
                return
            allreduce_packed(sums, counts)
        elif self._count_features.is_contiguous():
            # single process: the running-mean update rides on the finalize launch of the sums
            self.ready_flag = ops.proto_accumulate_update(features, task, rank, n_bt, mode, self._prototypes_tensors,
                                                          self._count_features)[2]
            return
        else:
            sums, counts = ops.proto_accumulate(features, task, rank, n_bt, T, mode)
        self.ready_flag = ops.proto_update(self._prototypes_tensors, self._count_features, sums, counts)

    def update_prototypes(self, model, img, target):
        features = model.get_penultimate_output(img)
        self.update_feats_prototypes(features, target)

    def _extract_labels_prototype_index(self, features, target, include_bg=False, labels_down=None):
        """Inspection helper with the reference's return shape (prototypes.py:177-205);
        synchronises (torch.unique) and is not used by update_feats_prototypes."""
        B, D, h, w = features.shape
        T = ops.MAX_TASKS
        lut = self._device_task_lut(features.device, T)
        labels = target if labels_down is None else labels_down.reshape(B, h, w)
        _, _, _, down = ops.label_downsample_task(labels.long(), h, w, lut, T, want_labels_down=True)
        down = down.unsqueeze(1)
        cl_present = torch.unique(down, sorted=True)
        if cl_present.numel() and cl_present[-1] == self.ignore_index:
            cl_present = cl_present[:-1]
        if int(((down != 0) & (down != self.ignore_index)).sum()) == 0:
            return None
        task_nums = {}
        current_tasks = np.broadcast_to(self.label_to_task_num(cl_present), (cl_present.numel(),))
        for idx, cl in enumerate(cl_present):
            if cl == 0 and not include_bg:
                continue
            task_nums.setdefault(int(current_tasks[idx]), []).append(cl)
        return features, D, down, task_nums

    def compute_loss(self, batch, model, train=True):
        """prototypes.py:207-229."""
        if isinstance(batch, dict):
            img, mask = batch["main"][0], batch["main"][1]
        else:
            img, mask = batch[0], batch[1]
        if train:
            self.update_prototypes(model, img, mask)
        loss, preds_mask = self.compute_base_loss(img, mask, model, train=train)
        return loss, self._argmax(preds_mask)
