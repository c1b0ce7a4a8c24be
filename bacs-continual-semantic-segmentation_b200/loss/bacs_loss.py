"""BACSLoss -- drop-in for the reference's ``loss.BACSLoss`` (loss/bacs_loss.py:14-463).

Same constructor keywords (conf/experiments/loss/bacs_plus.yaml), lifecycle hooks and
``compute_loss(batch, model, train) -> (loss, preds)`` contract.  Per training step
(task > 0, ``bg_weighted_ce``, ``lkd > 0``, replay on) the device executes, with no host
synchronisation in between:

  label down-sample + task/rank      csrc/labels.cu        (prototypes.py:177-205)
  prototype segmented reduction      csrc/prototypes.cu    (prototypes.py:127-163)
  seen head logits at stride 16      csrc/seen.cu          (bg_detector.py:17-40)
  fused pixel kernel                 csrc/pixel_loss.cu    (loss_utils.py:542-585,
        weighted CE + focal + arg-max + distill mask + dlogits   base_loss.py:255-272, bacs_loss.py:255,282-285)
  teacher distill fwd+bwd            csrc/distill.cu       (bacs_loss.py:258-294)
  replay: class-weighted CE (dark++) + prototype update on replay features (Q11)
          + DER logit MSE with transplant   csrc/misc.cu   (bacs_loss.py:342-431)"""
from __future__ import annotations

from copy import deepcopy as copy

import torch

from .. import ops
from ..autograd import DerMseFunction, TeacherDistillFunction, join_side_stream
from .base_loss import BaseLoss, SeenMap
from .experience_replay import ExperienceReplay


def freeze_network(model):
    """training/utils.py:33-36"""
    for par in model.parameters():
        par.requires_grad = False
    model.eval()


class BACSLoss(ExperienceReplay):
    def __init__(self, name="BACS", ignore_index=255, alpha: float = 0.8, beta: float = 0.2, buffer_size: int = 50,
                 replay_minibatch_size: int = 32, dark_plus_plus: bool = True, use_cosine_dist: bool = False,
                 same_task: bool = False, ignore_rep_bg: bool = True, bg_weighted_ce: bool = False,
                 seen_gamma: float = 2, seen_threshold: float = 0.5, seen_ukd: bool = True,
                 seen_focal_alpha: float = None, lkd: float = 0.25, lkd_alpha: float = 0.2,
                 lkd_threshold: float = 0.5, pseudo_label: bool = False, fused_logit_upsample: bool = False):
        super().__init__(name, ignore_index=ignore_index, same_task=same_task,
                         replay_minibatch_size=replay_minibatch_size, buffer_size=buffer_size,
                         bg_weighted_ce=bg_weighted_ce)
        self.alpha = alpha
        self.beta = beta
        self.fused_logit_upsample = bool(fused_logit_upsample)   # extra keyword (not in the reference), default off
        self.dark_plus_plus = dark_plus_plus
        self.use_cosine_dist = use_cosine_dist
        if use_cosine_dist:
            raise NotImplementedError("BACSLoss(use_cosine_dist=True): the CosineEmbeddingLoss variant "
                                      "(bacs_loss.py:75-78) is not on the benchmarked path")
        self._use_der_loss = False
        self.ignore_rep_bg = ignore_rep_bg
        self.buffer = None
        self.update_buffer_every = 1
        self.bg_weighted_ce = bg_weighted_ce
        self.prev_model = None
        self.init_weighted_loss(gamma=seen_gamma, threshold=seen_threshold, ukd=seen_ukd)
        self.lkd = lkd
        self.lkd_threshold = lkd_threshold
        self.lkd_alpha = lkd_alpha
        self.pseudo_label = pseudo_label and not bg_weighted_ce
        self.seen_focal_alpha = seen_focal_alpha
        self.init_seen_focal_loss(alpha=seen_focal_alpha)
        self.logit_transforms = lambda x: x
        self.dark_criterion = None

    def _init_dark_criterion(self, device):
        self.dark_criterion = "mse"

    # ---- lifecycle ------------------------------------------------------------------------------
    def _attach_replay_loaders(self, trainer, datamodule):
        """From the second task on the training loop iterates three loaders in lock-step (reference
        bacs_loss.py:97-124): the task's own batches, replayed (image, label) pairs and replayed (image, stored
        low-res logits, class count) triples, the latter with torchvision's RandomAutocontrast on the images."""
        from pytorch_lightning.trainer.supporters import CombinedLoader   # the caller's Lightning
        from torchvision import transforms as tv
        buf = self._get_current_buffer()
        autocontrast = tv.RandomAutocontrast(p=0.5)
        loaders = {
            "main": trainer.train_dataloader.loaders,
            "buffer": datamodule.get_buffer_loader(buf.img_paths, buf.target_paths, target_trsf=buf.target_trsf),
            "bufferlogits": datamodule.get_logits_loader(
                buf.dataset_map["examples"], buf.dataset_map["logits"], buf._logits_n_classes, length=len(buf.img_paths),
                transforms=tv.Compose([tv.Lambda(lambda x: torch.from_numpy(x)), autocontrast])),
        }
        trainer.train_dataloader = CombinedLoader(loaders, "max_size_cycle")
        self.logit_transforms = autocontrast

    def on_train_start(self, task_num, **kwargs):
        """Start of a task (reference bacs_loss.py:82-131): open the replay buffer for the task's class count, switch
        the replay terms on after the first task, and keep the teacher frozen on the training device."""
        self.accelerator = kwargs.get("accelerator")
        device = self.accelerator.root_device
        self._init_dark_criterion(device=device)
        self._init_buffer(task_num=task_num)
        self._iter_indx = 0
        self.update_buffer_every = kwargs.get("accumulate_grad_batches", 1)
        if task_num > 0:
            assert self.same_task is False
            self._use_der_loss = True
            datamodule = kwargs.get("datamodule")
            if datamodule is not None and (self.alpha > 0 or self.beta > 0):
                self._attach_replay_loaders(kwargs.get("trainer"), datamodule)
        if self.prev_model is not None:
            self.prev_model = self.prev_model.to(device)
            freeze_network(self.prev_model)

    @staticmethod
    def _train_set_files(loader, trainer):
        """(dataset, image paths, label paths) in loader order; sweeps / debug runs wrap the dataset in a Subset"""
        datamodule = getattr(trainer, "datamodule", None)
        if datamodule is not None and (getattr(datamodule, "_sweep", False) or getattr(datamodule, "debug", False)):
            subset = loader.dataset.base_dataset
            return subset.dataset, subset.dataset._x[subset.indices], subset.dataset._y[subset.indices]
        return loader.dataset, loader.dataset._x, loader.dataset._y

    def on_train_end(self, **kwargs):
        """End of a task (reference bacs_loss.py:133-203): the trained model becomes the frozen teacher, then one
        un-shuffled pass over the task's training set offers every image to the replay buffer together with its
        low-res logits, the importance score (SCORE mode of the fused kernel), the seen map and its file paths."""
        BaseLoss.on_train_end(self, **kwargs)
        if not kwargs.get("pre_last_tasks"):
            return
        model, loader = kwargs.get("model"), kwargs.get("train_dataloader")
        if self.buffer is None:
            self._init_buffer()
        self.prev_model = model.clone()
        freeze_network(self.prev_model)
        if model is None or loader is None or not (self.alpha > 0 or self.beta > 0):
            return
        accelerator = kwargs.get("accelerator")
        device = accelerator.root_device
        model = model.to(device)
        loader.shuffle = False
        dataset, images_on_disk, labels_on_disk = self._train_set_files(loader, kwargs.get("trainer"))
        class_w = torch.ones(self.nb_current_classes, device=device)
        class_w[0] = 0
        seen = 0
        with torch.no_grad():
            for batch in accelerator.process_dataloader(loader):
                images, labels = accelerator.to_device(batch)[:2]
                labels = labels.long()
                files = slice(seen, seen + images.shape[0])
                model.enable_caching_sem_logits()
                score = self._score_batch(model, images, labels, class_w)[1]
                self._add_to_buffer(images, model.pop_sem_logits(), labels, score,
                                    seen_detector=self._get_seen_detector(images, model), paths=images_on_disk[files],
                                    target_paths=labels_on_disk[files], target_trsf=copy(dataset.target_trsf))
                seen = files.stop
        self.update_buffer_scores()

    # ---- step ------------------------------------------------------------------------------------
    def post_process_mask(self, img, mask):
        """bacs_loss.py:205-210: optional pseudo-labelling of background by the old model, in place on ``mask`` by one
        kernel (no host synchronisation).  With ``fused_logit_upsample`` the teacher's low-res sem_logits are read and
        the pseudo labels follow that flag's arg-max contract (identical except at fp32 near-ties)."""
        if self.pseudo_label and self.prev_model is not None:
            with torch.no_grad():
                if self.fused_logit_upsample:
                    ops.pseudo_label_inplace(mask, self.prev_model(img, return_sem_logits=True), lowres=True)
                else:
                    ops.pseudo_label_inplace(mask, self.prev_model(img))
        return mask

    def compute_loss(self, batch, model, train=True):
        """bacs_loss.py:212-256."""
        if isinstance(batch, dict):
            img, mask = batch["main"][0], batch["main"][1]
        else:
            img, mask = batch[0], batch[1]
        if train:
            mask = self.post_process_mask(img, mask)
        with_distill = self._use_der_loss and train and self.lkd > 0
        out = self.compute_base_loss(img, mask, model, train=train,
                                     use_weighted_ce=self.bg_weighted_ce and self._use_der_loss,
                                     return_attentions=with_distill)
        if with_distill:
            loss, preds_mask, old_attention, new_attention, seen_prob = out
            loss = self._teacher_distill(old_attention, new_attention, seen_prob, mask, _add_to=loss)
        else:
            loss, preds_mask = out
        preds_output = self._argmax(preds_mask)        # produced by the fused kernel, no second read
        if train and self._use_der_loss and (self.alpha > 0 or self.beta > 0):
            loss = loss + self._replay_der_loss(model, batch["buffer"], batch["bufferlogits"])
        join_side_stream()      # the seen-head backward forked by the pixel-loss op ran next to the distill chain
        return loss, preds_output

    def _teacher_distill(self, old_attention, new_attention, seen_prob, mask, _add_to=None):
        """bacs_loss.py:258-294.  ``seen_prob`` is the SeenMap handle produced by
        compute_base_loss (its distill mask came out of the fused pixel kernel), a plain
        [B,T,H,W] probability tensor, or None.  ``_add_to`` (not in the reference): a loss tensor the term is added
        to by the kernel's own reduction launch; the sum is returned."""
        if self.lkd == 0:
            return 0 if _add_to is None else _add_to
        if isinstance(seen_prob, SeenMap) and seen_prob.distill_mask is not None:
            m = seen_prob.distill_mask
        elif seen_prob is None and self._fused_distill_mask is not None \
                and self._fused_distill_mask.shape == mask.shape:
            m = self._fused_distill_mask
        else:
            m = mask == 0
            if seen_prob is not None:
                probs = seen_prob.materialize() if isinstance(seen_prob, SeenMap) else seen_prob
                m = m & (probs.max(1)[0] > self.lkd_threshold)
            m = m.to(torch.uint8)
        fuse = (_add_to is not None and torch.is_tensor(_add_to) and _add_to.is_cuda and _add_to.dtype == torch.float32
                and _add_to.numel() == 1)
        term = TeacherDistillFunction.apply(new_attention[-1], old_attention[-1], m, tuple(mask.shape[-2:]),
                                            float(self.lkd), _add_to if fuse else None)
        return term if (fuse or _add_to is None) else _add_to + term

    def _get_seen_detector(self, img, model, task_num=-1):
        """bacs_loss.py:296-306: full-res seen logits of one head (buffer population)."""
        seen_net = getattr(model, "seen_fg_network", None)
        if seen_net is None:
            return None
        pen = model.get_penultimate_output(img)
        protos = self.prototypes
        head = task_num if task_num >= 0 else protos.shape[0] + task_num
        heads = self._heads(seen_net)
        mod = heads[head] if len(heads) > 1 else heads[0]
        z = ops.seen_logits(pen.detach(), protos[head:head + 1], mod.conv.weight.detach().reshape(1, -1),
                            mod.conv.bias.detach().reshape(1))
        return ops.seen_upsample(z, 16, apply_sigmoid=False)

    def _add_to_buffer(self, examples, logits, labels, losses, seen_detector=None, paths=None, target_paths=None,
                       target_trsf=None):
        """bacs_loss.py:308-340."""
        with torch.no_grad():
            new_data = {"examples": examples.detach().cpu(), "logits": logits.detach().float().cpu(),
                        "labels": labels.cpu(), "loss": losses.detach().cpu(), "img_paths": paths,
                        "target_paths": target_paths, "target_trsf": [target_trsf for _ in range(len(paths))]}
            if seen_detector is not None:
                new_data["seen"] = seen_detector.detach().cpu()
            self._get_current_buffer().add_data(new_data)

    # ---- replay ------------------------------------------------------------------------------------
    def _dark_pp(self, model, memory_data, _scale=1.0):
        """bacs_loss.py:342-385: class-weighted CE on replay images; also moves the prototypes
        with the replay features (Q11).  The mix-up branch needs 'lamdas' in the batch, which
        no loader of the reference produces."""
        if memory_data is None or not self.dark_plus_plus:
            return 0
        memory_dict, memory_inputs, _, memory_labels, _, _ = memory_data
        if "lamdas" in memory_dict:
            raise NotImplementedError("BACSLoss._dark_pp: the co-occurrence mix-up branch (bacs_loss.py:356-374)")
        classes_weights = torch.zeros(self.nb_current_classes, device=self.device)
        classes_weights[(1 if self.ignore_rep_bg else 0):self.old_classes] = 1
        loss, _ = self.compute_base_loss(memory_inputs.float(), memory_labels.long(), model, task_num=None,
                                         weights=classes_weights, train=True, use_weighted_ce=False,
                                         _loss_scale=_scale)
        return loss

    def _dark_logits(self, model, memory_data, _scale=1.0):
        """bacs_loss.py:387-431: MSE between the stored (int-truncated, Q4) logits with the
        reference's single-sample transplant (Q5) and the live low-res logits."""
        if memory_data is None:
            return 0
        _, memory_inputs, memory_logits, _, n_classes_per_logit, _ = memory_data
        memory_inputs = self.logit_transforms(memory_inputs)
        sem_logits = model(memory_inputs, return_sem_logits=True)
        if self.same_task:
            raise NotImplementedError("BACSLoss(same_task=True) is asserted off by the reference (bacs_loss.py:95)")
        cut = ops.der_cut(n_classes_per_logit.to(sem_logits.device), sem_logits.shape[1])
        return DerMseFunction.apply(sem_logits, memory_logits, cut, bool(self.ignore_rep_bg), True, float(_scale))

    def _replay_der_loss(self, model, replay_batch=None, replay_logits=None):
        """bacs_loss.py:433-463: beta * dark++ + alpha * dark logits (weights folded into the kernels)."""
        loss = 0
        if self.beta != 0:
            data = ({"examples": replay_batch[0], "labels": replay_batch[1]}, replay_batch[0], None,
                    replay_batch[1], None, None)
            loss = loss + self._dark_pp(model, data, _scale=self.beta)
        if self.alpha != 0:
            data = ({"examples": replay_logits[0], "labels": None}, replay_logits[0], replay_logits[1], None,
                    replay_logits[2], None)
            loss = loss + self._dark_logits(model, data, _scale=self.alpha)
        return loss
