"""The DeepLabV3+/WideResNet38 harness trunk (harness/deeplab_wrn38.py) keeps the reference's checkpoint layout and block
names: key/shape listing frozen from models/deeplabv3/deeplabv3.py:DeepWV3Plus (tests/golden/deepwv3plus_keys.json, written
by oracle/make_golden_steps.py), the survey's parameter-count known answers, and the 51M plan's surgery through the
drop-in student wrapper, and the forward pass against stored outputs of the reference class
(tests/golden/deepwv3plus_forward.npz)."""
import json
import os

import numpy as np
import pytest
import torch

import kdcc
from conftest import GOLDEN
from harness.deeplab_wrn38 import DeepWV3Plus, PRUNING_51M, pruning_section


@pytest.fixture(scope="module")
def trunk():
    torch.manual_seed(0)
    return DeepWV3Plus(19).eval()


def test_state_dict_layout_matches_the_reference_class(trunk):
    want = json.load(open(os.path.join(GOLDEN, "deepwv3plus_keys.json")))
    have = {k: list(v.shape) for k, v in trunk.state_dict().items()}
    assert list(have) == list(want) and have == want
    assert sum(p.numel() for p in trunk.parameters()) == 137_103_936          # BASELINE.md: 137.10 M


def test_51m_plan_surgery_gives_the_survey_parameter_counts(trunk):
    from kdcc.trainer import prepare_train_epoch
    model = kdcc.DepthwiseStudent(trunk, {"trainer": {"verbosity": 2}})
    opt = prepare_train_epoch(model, pruning_section(), 1, None, lambda ps: torch.optim.SGD(ps, lr=0.1))
    assert model.replaced_block_names == PRUNING_51M["names"]
    sites = [(model.get_block(n, model.student).separable_conv.in_channels, model.get_block(n, model.student).pointwise_conv.out_channels)
             for n in PRUNING_51M["names"]]
    assert sites == [(512, 512)] * 5 + [(1024, 2048)] + [(4096, 256)] * 3       # what bench.py's PLAN_51M times
    assert sum(p.numel() for p in model.student.parameters()) == 85_960_768     # BASELINE.md: 85.96 M student
    assert sum(p.numel() for p in opt.param_groups[0]["params"]) == 7_839_232   # BASELINE.md: trainable
    assert not model.student.training                                            # F9: the student stays in eval mode


def test_forward_matches_the_reference_class(trunk):
    # deepwv3plus_forward.npz: the reference class's output on this input and these weights (oracle/make_golden_steps.py).
    # CPU convolutions pick their summation order by thread count and ISA: values 1e-6 of max |y| apart, channel sums
    # 2e-8 of the largest absolute sum.  The bounds keep a 10x margin over that; a BatchNorm eps of 1e-3 instead of 1e-5
    # in one middle unit moves the channel sums by 6e-7.
    g = np.load(os.path.join(GOLDEN, "deepwv3plus_forward.npz"))
    x = torch.randn(1, 3, 64, 96, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        y = trunk(x).numpy()
    assert list(y.shape) == g["shape"].tolist()
    np.testing.assert_allclose(y.reshape(-1)[g["idx"]], g["values"], rtol=0, atol=1e-5 * float(np.abs(g["values"]).max()))
    y64 = y.astype(np.float64)
    np.testing.assert_allclose(y64.sum(axis=(0, 2, 3)), g["channel_sum"], rtol=0, atol=2e-7 * float(g["channel_abs_sum"].max()))
    np.testing.assert_allclose(np.abs(y64).sum(axis=(0, 2, 3)), g["channel_abs_sum"], rtol=2e-7)
