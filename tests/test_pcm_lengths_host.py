"""CPU: DeployModel.frame_counts, the frame rule of forward(lengths=) and of the decoders' lens, without a device."""
from types import SimpleNamespace

import numpy as np
import torch

from keyword_spotting_b200 import Config, DeployModel
from oracle import model as om

LENGTHS = [0, 3, 399, 400, 401, 559, 560, 719, 720, 5360, 5521, 16000]


def _counts(lengths):
    return DeployModel.frame_counts(SimpleNamespace(config=Config()), lengths)


def test_frame_counts_follow_the_frame_rule():
    want = [max(0, om.num_frames(n)) for n in LENGTHS]
    assert _counts(LENGTHS) == want
    assert want[:6] == [0, 0, 0, 1, 1, 1] and want[6] == 2


def test_frame_counts_keep_the_container_type():
    want = [max(0, om.num_frames(n)) for n in LENGTHS]
    assert isinstance(_counts(LENGTHS), list)
    assert _counts(tuple(LENGTHS)) == tuple(want)
    assert _counts(560) == 2 and isinstance(_counts(560), int)
    a = _counts(np.array(LENGTHS, np.int32))
    assert isinstance(a, np.ndarray) and a.tolist() == want
    t = _counts(torch.tensor(LENGTHS, dtype=torch.int64))
    assert isinstance(t, torch.Tensor) and t.tolist() == want
