"""CPU: the host-side checks of export_streams / import_streams (ids and records), without a device."""
import numpy as np
import pytest
import torch

from keyword_spotting_b200 import InvalidArgumentError
from keyword_spotting_b200.streaming import record_ids, record_input


@pytest.mark.parametrize("ids,distinct", [([5], False), ([-1], False), ([1.0], False), ([[1]], False),
                                          (np.array([True]), False), ([2, 3, 2], True)],
                         ids=["past_end", "negative", "float", "2d", "bool", "duplicate"])
def test_invalid_host_ids_raise(ids, distinct):
    with pytest.raises(InvalidArgumentError):
        record_ids(ids, 5, None, distinct)


@pytest.mark.parametrize("records", [np.zeros((2, 16), np.int8), torch.zeros(3, 16, dtype=torch.uint8),
                                     np.zeros(31, np.uint8), torch.zeros(2, 16, dtype=torch.int32)],
                         ids=["int8", "rows", "bytes", "int32"])
def test_records_of_wrong_type_or_size_raise(records):
    with pytest.raises(InvalidArgumentError):
        record_input(records, 2, 16, None)
