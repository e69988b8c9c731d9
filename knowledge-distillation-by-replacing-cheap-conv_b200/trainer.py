"""The layerwise distillation step: loop body of trainer/layerwise_trainer.py:220-250, made sync-free and
data-parallel.

What is kept from the reference: `model(data)` -> (student, teacher) logits with hint features collected
by the hooks; supervised / KD / teacher losses computed for logging; the hint loss (sum over the hooked
pairs, divided by accumulation_steps) is the ONLY loss back-propagated (layerwise_trainer.py:229-235);
the optimizer steps when `batch_idx % accumulation_steps == 0` (so also on index 0, as in the reference).

What changes: no `.item()`, no `.cpu()` of the logits, no NumPy confusion matrix in the step (SURVEY.md
F13) -- losses stay 0-dim device tensors and the IoU confusion matrix is accumulated on the GPU; with
world_size > 1 the trainable student gradients are averaged with ONE all-reduce of a flat bucket (frozen
teacher replicated, eval-mode BN: no other cross-rank coupling, SURVEY.md 8e).
"""
from functools import reduce

import torch

from .metrics import ConfusionMatrix  # noqa: F401  (kernel-backed; kept importable from here)
from . import functional as F_kdcc
from .losses import CrossEntropyLoss2d, KLDivergenceLoss, MSELoss
import torch.distributed as dist


class GradBucket:
    """Flat fp32 view of the trainable parameters' gradients: one exchange per optimizer step.
    Rebuild it (`GradBucket(params)`) whenever prepare_train_epoch changes the trainable set.

    `peer=True` (CUDA, world > 1, kdcc.optim.RAdam): the bucket lives in a symmetric buffer (kdcc.PeerGradBucket); every
    parameter's gradient is pushed to the peers by copy engines the moment autograd has finished accumulating it, and the
    optimizer averages the ranks' copies inside its fused pass -- no collective kernel on the step's critical path.
    Otherwise: one NCCL (or gloo) all-reduce after the backward."""

    ALIGN = 32  # floats

    def __init__(self, params, peer=False, group=None, optimizer=None, push_in_backward=True):
        self.params = [p for p in params if p.requires_grad]
        # every gradient starts on a 128-byte boundary of the bucket (32 floats): the fused optimizer and the GEMM
        # epilogues use 16-byte accesses, and a 19-element classifier bias must not misalign whatever follows it
        self.offsets, off = [], 0
        for p in self.params:
            self.offsets.append(off)
            off += -(-p.numel() // self.ALIGN) * self.ALIGN
        dev = self.params[0].device if self.params else torch.device("cpu")
        self.peer, self._hooks, self._pushed = None, [], False
        if peer and self.params and dev.type == "cuda" and dist.is_available() and dist.is_initialized() and \
                dist.get_world_size(group) > 1 and hasattr(optimizer, "attach_grad_sources"):
            from .peer_reduce import PeerGradBucket
            try:
                self.peer = PeerGradBucket(off, dev, group)
            except Exception as exc:   # no symmetric memory on this system: every rank falls back to the all-reduce alike
                import warnings
                warnings.warn("kdcc.GradBucket: peer gradient exchange unavailable (%r); using the NCCL all-reduce" % (exc,))
                self.peer = None
        if self.peer is not None:
            self.flat = self.peer.local()
            for p, o in zip(self.params, self.offsets):
                optimizer.attach_grad_sources(p, lambda o=o, n=p.numel(): (self.peer.sources()[0][o:o + n],) + self.peer.sources()[1:])
                if push_in_backward:
                    self._hooks.append(p.register_post_accumulate_grad_hook(
                        lambda prm, o=o, n=p.numel(): self._push(o, o + n)))
        else:
            self.flat = torch.zeros(off, dtype=torch.float32, device=dev)
            for p in self.params:   # a bucket rebuilt without the peer exchange must not leave stale sources behind
                getattr(optimizer, "_sources", {}).pop(p, None)
        self._point_grads()

    def _point_grads(self):
        for p, o in zip(self.params, self.offsets):  # .grad become views into the bucket: no copies at step time
            p.grad = self.flat[o:o + p.numel()].view_as(p)

    def _push(self, lo, hi):
        self.peer.push(lo, hi)
        self._pushed = True

    def zero(self):
        """After the optimizer step: == optimizer.zero_grad() for the trainable set, keeps the flat views alive."""
        if self.peer is not None:   # the next step fills the other parity of the symmetric buffer
            self.peer.flip()
            self.flat = self.peer.local()
            self._point_grads()
            self._pushed = False
        self.flat.zero_()

    def dense(self):
        """The gradients back to back without the alignment padding (a copy; for tests and logging)."""
        return torch.cat([self.flat[o:o + p.numel()] for p, o in zip(self.params, self.offsets)]) if self.params else self.flat

    def all_reduce_mean(self, group=None):
        """Make the rank-averaged gradient available to the optimizer step that follows."""
        if self.peer is not None:
            if not self._pushed:                 # nothing went out during the backward (hooks off, or gradient accumulation)
                self.peer.push(0, self.peer.numel)
            self.peer.finish()
            return
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            world = dist.get_world_size(group)
            if dist.get_backend(group) == "nccl":
                dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=group)
            else:  # gloo has no AVG
                dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)
                self.flat.div_(world)

    def close(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []


def _expect(criterion, value):
    """Tell a kdcc criterion which upstream gradient its backward will see (a device-verified performance hint, see
    kdcc.losses); anything that is not a kdcc criterion is left alone."""
    if hasattr(criterion, "expected_upstream"):
        criterion.expected_upstream = float(value)


def _confusion_of(metric):
    """(int64 C*C device matrix, ignore_index) behind a ConfusionMatrix / CityscapesMetricTracker."""
    cm = getattr(metric, "_cm", metric)
    return cm.mat, cm.ignore


class LayerwiseStep:
    """criterions = [supervised, kd, hint] as in train.py:48-50; `model` is a DepthwiseStudent.

    `metrics` (optional): a (student, teacher) pair of kdcc ConfusionMatrix / CityscapesMetricTracker updated with the
    step's logits (trainer/layerwise_trainer.py:247-250).  When criterions[0] is a kdcc CrossEntropyLoss2d, the logged
    supervised / teacher CE, the KD term (kdcc KLDivergenceLoss or MSELoss; any other criterion is called as it is) and
    both confusion matrices come from ONE pass over the two logit tensors and the labels (kdcc_logits_stats)."""

    def __init__(self, model, criterions, optimizer, accumulation_steps=1, process_group=None, log_supervised=True,
                 peer_exchange=True, metrics=None):
        self.model, self.criterions, self.optimizer = model, criterions, optimizer
        self.accumulation_steps = int(accumulation_steps)
        self.group = process_group
        self.log_supervised = log_supervised
        self.peer_exchange = peer_exchange
        self.metrics = metrics
        self.bucket = None
        self.rebuild_bucket()
        _expect(criterions[2], 1.0 / self.accumulation_steps)   # loss = sum(hint pairs) / accumulation_steps

    def rebuild_bucket(self):
        if self.bucket is not None:
            self.bucket.close()
        # gradients leave for the peers while the backward is still running only when every backward ends in a step
        self.bucket = GradBucket(self.model.trainable_parameters(), peer=self.peer_exchange, group=self.group,
                                 optimizer=self.optimizer, push_in_backward=self.accumulation_steps == 1)

    def __call__(self, data, target, batch_idx):
        acc = self.accumulation_steps
        output_st, output_tc = self.model(data)
        pairs = list(zip(self.model.student_hidden_outputs, self.model.teacher_hidden_outputs))
        hint_loss = reduce(lambda a, st: a + self.criterions[2](st[0], st[1]), pairs, 0) / acc
        with torch.no_grad():  # logged, never back-propagated by this trainer
            if self.log_supervised and target is not None and isinstance(self.criterions[0], CrossEntropyLoss2d):
                kd_loss, supervised, teacher_loss = self._fused_stats(output_st, output_tc, target)
            else:
                kd_loss = self.criterions[1](output_st, output_tc) / acc
                if self.log_supervised and target is not None:
                    supervised = self.criterions[0](output_st, target) / acc
                    teacher_loss = self.criterions[0](output_tc, target)
                else:
                    supervised = teacher_loss = torch.zeros((), device=data.device)
                if self.metrics is not None and target is not None:
                    self.metrics[0].update(output_st, target)
                    self.metrics[1].update(output_tc, target)
        loss = hint_loss
        if torch.is_tensor(loss):
            loss.backward()
        if batch_idx % acc == 0:
            self.bucket.all_reduce_mean(self.group)
            self.optimizer.step()
            self.bucket.zero()  # == optimizer.zero_grad() for the trainable set, keeps the flat views alive
        return {"loss": loss, "hint_loss": hint_loss, "kd_loss": kd_loss, "supervised_loss": supervised,
                "teacher_loss": teacher_loss, "output_st": output_st.detach(), "output_tc": output_tc}

    def _fused_stats(self, output_st, output_tc, target):
        """(kd / acc, supervised / acc, teacher) of one kdcc_logits_stats pass; confusion matrices that do not share the
        criterion's ignore_index or class count are updated by their own pass."""
        acc = self.accumulation_steps
        ce, kd_crit = self.criterions[0], self.criterions[1]
        kd_mode, T, scale = 0, 1.0, 1.0
        if isinstance(kd_crit, KLDivergenceLoss):
            kd_mode, T = 1, float(kd_crit.temperature)
        elif isinstance(kd_crit, MSELoss):
            kd_mode, scale = 2, float(kd_crit.num_classes)
        confs, separate = [None, None], []
        for i, (metric, logits) in enumerate(zip(self.metrics or (), (output_st, output_tc))):
            mat, ignore = _confusion_of(metric)
            if ignore == ce.ignore_index and mat.numel() == logits.shape[1] ** 2:
                confs[i] = mat
            else:
                separate.append((metric, logits))
        kd, sup, tea = F_kdcc.logits_stats(output_st, output_tc, target, ce.weight, ce.ignore_index,
                                           mean=ce.size_average is not False, kd_mode=kd_mode, temperature=T, kd_scale=scale,
                                           conf_s=confs[0], conf_t=confs[1])
        for metric, logits in separate:
            metric.update(logits, target)
        kd_loss = (kd if kd_mode else kd_crit(output_st, output_tc)) / acc
        return kd_loss, sup / acc, tea


class ClassificationStep:
    """Loop body of trainer/classification_trainer.py:24-43 (the CIFAR-10 configs, train_classification.py): the same
    forward and the same three criterions as the layerwise loop, but the loss that is back-propagated is the KD term
    (`loss = kd_loss`, :38-39) and the optimizer steps when `(batch_idx + 1) % accumulation_steps == 0` (:41-43 -- not
    on index 0, unlike the layerwise loop).  Supervised, hint and teacher losses are computed for logging only, as
    0-dim device tensors (no `.item()` in the step).  Note: this trainer keeps the student in train mode, so its
    BatchNorm statistics are per rank under data parallelism (the reference runs it on one device)."""

    def __init__(self, model, criterions, optimizer, accumulation_steps=1, process_group=None):
        self.model, self.criterions, self.optimizer = model, criterions, optimizer
        self.accumulation_steps = int(accumulation_steps)
        self.group = process_group
        self.bucket = GradBucket(model.trainable_parameters())
        _expect(criterions[1], 1.0 / self.accumulation_steps)   # loss = kd / accumulation_steps

    def rebuild_bucket(self):
        self.bucket = GradBucket(self.model.trainable_parameters())

    def __call__(self, data, target, batch_idx):
        acc = self.accumulation_steps
        output_st, output_tc = self.model(data)
        kd_loss = self.criterions[1](output_st, output_tc) / acc
        with torch.no_grad():  # logged, never back-propagated by this trainer
            supervised = self.criterions[0](output_st, target) / acc
            pairs = zip(self.model.student_hidden_outputs, self.model.teacher_hidden_outputs)
            hint_loss = reduce(lambda a, st: a + self.criterions[2](st[0], st[1]), pairs, torch.zeros((), device=data.device)) / acc
            teacher_loss = self.criterions[0](output_tc, target)
        loss = kd_loss
        loss.backward()
        if (batch_idx + 1) % acc == 0:
            self.bucket.all_reduce_mean(self.group)
            self.optimizer.step()
            self.bucket.zero()
        return {"loss": loss, "hint_loss": hint_loss, "kd_loss": kd_loss, "supervised_loss": supervised,
                "teacher_loss": teacher_loss, "output_st": output_st.detach(), "output_tc": output_tc}


class EnsembleStep:
    """Loop body of trainer/ensemble_trainer.py:73-90 (multi-teacher distillation, BASELINE config 5): the student is
    distilled from its own teacher and from `models` (other, frozen, students), with
        kd = (sum_k WEIGHT * crit_kd(student, model_k(x)) + crit_kd(student, teacher)) / (WEIGHT * K + 1)
    and `loss = kd + supervised`, both divided by accumulation_steps; step on `(batch_idx + 1) % accumulation_steps`.
    `kd_multi` (a kdcc.MultiTeacherKLDivergenceLoss) computes the whole KD term in one fused pass -- student logits read
    once, every teacher once; without it the term is composed from criterions[1] exactly as the reference composes it."""

    def __init__(self, model, models, criterions, optimizer, accumulation_steps=1, weight=1, kd_multi=None, process_group=None):
        self.model, self.models, self.criterions, self.optimizer = model, list(models), criterions, optimizer
        self.accumulation_steps, self.weight, self.kd_multi = int(accumulation_steps), weight, kd_multi
        self.group = process_group
        self.bucket = GradBucket(model.trainable_parameters())
        _expect(criterions[0], 1.0 / self.accumulation_steps)   # loss = kd + supervised / accumulation_steps

    def rebuild_bucket(self):
        self.bucket = GradBucket(self.model.trainable_parameters())

    def __call__(self, data, target, batch_idx):
        acc = self.accumulation_steps
        output_st, output_tc = self.model(data)
        with torch.no_grad():
            outputs = [m(data) for m in self.models]
        supervised = self.criterions[0](output_st, target) / acc
        if self.kd_multi is not None:
            kd_loss = self.kd_multi(output_st, outputs, output_tc) / acc
        else:
            kd_loss = reduce(lambda a, o: a + self.weight * self.criterions[1](output_st, o), outputs, 0)
            kd_loss = (kd_loss + self.criterions[1](output_st, output_tc)) / (self.weight * len(outputs) + 1) / acc
        loss = kd_loss + supervised
        loss.backward()
        if (batch_idx + 1) % acc == 0:
            self.bucket.all_reduce_mean(self.group)
            self.optimizer.step()
            self.bucket.zero()
        return {"loss": loss, "kd_loss": kd_loss, "supervised_loss": supervised, "output_st": output_st.detach(),
                "output_tc": output_tc}


def prepare_train_epoch(model, pruning, epoch, optimizer, make_optimizer, optimizer_args=None, step=None):
    """Epoch-boundary surgery of trainer/layerwise_trainer.py:78-150 (+ update_optimizer :152-175, create_new_optimizer
    :177-186) for a kdcc.DepthwiseStudent.  `pruning` is the config's "pruning" section (`pruning_plan`, `hint`,
    `unfreeze` lists of {"name", "epoch", ...} and `args`, the default block geometry; `pruner` in old checkpoints).

    * epoch 1 with three empty lists: the whole student becomes trainable and gets a fresh optimizer;
    * an epoch that no list mentions changes nothing;
    * otherwise the blocks of this epoch are replaced, hooked and unfrozen; epoch 1 builds a NEW optimizer over the
      trainable student parameters (`make_optimizer(params)`), later epochs add one param group per unfrozen layer
      with `optimizer_args` (+ the layer's own "lr").  As in the reference the "lr" override is written INTO
      `optimizer_args` (:171-172), so it also applies to the layers that follow without an "lr" of their own (pass
      the config's optimizer "args" dict; with None the dict is kept on the model so the override still persists).
    Returns the optimizer to use from now on; a LayerwiseStep passed as `step` gets it and rebuilds its flat gradient
    bucket (the trainable set changed, SURVEY.md 8e)."""
    plan, hint, unfreeze = pruning['pruning_plan'], pruning['hint'], pruning['unfreeze']

    def done(opt):
        if step is not None:
            step.optimizer = opt
            step.rebuild_bucket()
        return opt

    if epoch == 1 and len(plan) + len(hint) + len(unfreeze) == 0:
        for prm in model.student.parameters():
            prm.requires_grad = True
        return done(make_optimizer([prm for prm in model.student.parameters() if prm.requires_grad]))
    if epoch not in [x['epoch'] for x in plan + hint + unfreeze]:
        return optimizer
    now = lambda entries: [x for x in entries if x['epoch'] == epoch]
    kwargs = pruning['args'] if 'args' in pruning else pruning['pruner']
    model.replace(now(plan), **kwargs)
    model.register_hint_layers([x['name'] for x in now(hint)])
    model.unfreeze([x['name'] for x in now(unfreeze)])
    if epoch == 1:
        return done(make_optimizer([prm for prm in model.student.parameters() if prm.requires_grad]))
    if optimizer_args is None:
        # the reference mutates config['optimizer']['args'] itself, so an "lr" override outlives the epoch; without a
        # caller-owned dict the same persistence is kept on the model
        optimizer_args = model.__dict__.setdefault('_kdcc_optimizer_args', {})
    for entry in now(unfreeze):
        layer = model.get_block(entry['name'], model.student)
        if 'lr' in entry:
            optimizer_args['lr'] = entry['lr']
        optimizer.add_param_group({'params': list(layer.parameters()), **optimizer_args})
    return done(optimizer)
