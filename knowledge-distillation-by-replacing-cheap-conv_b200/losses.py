"""Teacher->student distillation losses on libkdcc: same class names, constructor arguments and
call signatures as the reference's `losses` package, so `getattr(losses, cfg['kd_loss']['type'])(**args)`
(parse_config.py:89-93, train.py:48-50) keeps working.  Each forward is ONE fused kernel pass that
also emits the gradient; the result is a 0-dim fp32 tensor with a grad_fn.
"""
from torch import nn

from . import functional as F_kdcc

# Every criterion carries `expected_upstream` (default 1.0): the value its backward expects from autograd -- 1 for
# `loss.backward()`, 1 / accumulation_steps inside the layerwise loop (kdcc.LayerwiseStep sets it).  It is folded into the
# gradient the fused forward kernel emits and verified on the device in backward (rescaled there if it turns out to
# differ), which removes a full read-modify-write pass over the gradient from every backward.  Not a reference argument.


class CrossEntropyLoss2d(nn.Module):
    """losses/CrossEntropy.py:7-15 -- NLLLoss2d(log_softmax(inputs, 1), weight, size_average, ignore_index): weighted mean
    (size_average True or None) or sum of the per-pixel NLL over the pixels whose label is not ignore_index.  The value
    and the gradient come from one kernel pass; labels outside [0, C) other than ignore_index are dropped instead of
    stopping the device."""

    def __init__(self, weight=None, size_average=True, ignore_index=255):
        super().__init__()
        self.register_buffer("weight", weight)   # as NLLLoss2d: follows the module to the device
        self.size_average = size_average
        self.ignore_index = ignore_index
        self.expected_upstream = 1.0

    def forward(self, inputs, targets):
        return F_kdcc.cross_entropy(inputs, targets, self.weight, self.ignore_index, mean=self.size_average is not False,
                                    expected_upstream=self.expected_upstream)


class KLDivergenceLoss(nn.Module):
    """losses/KLDiv.py:4-23 -- kl_div(log_softmax(s/T), softmax(t/T)) * T^2 * C, 'mean' over all elements."""

    def __init__(self, temperature=1):
        super().__init__()
        self.temperature = temperature
        self.expected_upstream = 1.0

    def forward(self, inputs, targets):
        return F_kdcc.kd_loss(inputs, targets, self.temperature, target_is_prob=False, expected_upstream=self.expected_upstream)


class EnsembleKLDivergenceLoss(nn.Module):
    """losses/EnsembleKLDiv.py:5-22 -- targets are already probabilities (soft ensemble prediction)."""

    def __init__(self):
        super().__init__()
        self.expected_upstream = 1.0

    def forward(self, inputs, targets):
        return F_kdcc.kd_loss(inputs, targets, 1.0, target_is_prob=True, expected_upstream=self.expected_upstream)


class MSELoss(nn.Module):
    """losses/MSELoss.py:4-16 -- nn.MSELoss(reduction) * num_classes."""

    def __init__(self, reduction='mean', num_classes=19):
        super().__init__()
        if reduction != 'mean':
            raise ValueError("kdcc MSELoss implements reduction='mean' (the only value the reference configs use)")
        self.reduction = reduction
        self.num_classes = num_classes
        self.expected_upstream = 1.0

    def forward(self, inputs, targets):
        return F_kdcc.hint_loss(inputs, targets, None, scale=float(self.num_classes), expected_upstream=self.expected_upstream)


class WeightedHintMSELoss(nn.Module):
    """losses/WeightedHintMSELoss.py:5-16 -- per-channel weighted spatial-mean squared difference.
    `reduction` / `num_classes` are stored and unused, exactly as in the reference."""

    def __init__(self, reduction='mean', num_classes=19):
        super().__init__()
        self.reduction = reduction
        self.num_classes = num_classes
        self.expected_upstream = 1.0

    def forward(self, inputs, targets, filter_weight):
        return F_kdcc.hint_loss(inputs, targets, filter_weight, scale=1.0, expected_upstream=self.expected_upstream)


class MultiTeacherKLDivergenceLoss(nn.Module):
    """The KD term of trainer/ensemble_trainer.py:76-83 as one module:
        (sum_k WEIGHT * KL_T(student, ensemble_k) + KL_T(student, teacher)) / (WEIGHT * K + 1)
    with every KL a losses/KLDiv.py KLDivergenceLoss(temperature).  One fused pass reads the student logits once and
    each teacher once (kdcc_kd_loss_multi) instead of K + 1 criterion calls."""

    def __init__(self, temperature=1, weight=1):
        super().__init__()
        self.temperature = temperature
        self.weight = weight  # WEIGHT of trainer/ensemble_trainer.py:10
        self.expected_upstream = 1.0

    def forward(self, inputs, ensemble_outputs, teacher_output=None):
        outs = list(ensemble_outputs)
        w = [float(self.weight)] * len(outs)
        if teacher_output is not None:
            outs.append(teacher_output)
            w.append(1.0)
        total = sum(w)
        return F_kdcc.kd_loss_multi(inputs, outs, [x / total for x in w], self.temperature, expected_upstream=self.expected_upstream)
