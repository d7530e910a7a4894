"""CPU: the live session's host-side slot-list validation (septfa_b200.live.check_slots), which refuses a bad list with
ValueError before the library is called."""
import numpy as np
import pytest
import torch

from septfa_b200.live import check_slots


def test_check_slots_accepts_distinct_in_range_lists_in_any_order():
    for slots in ([3], [2, 0, 3], np.array([1, 0], dtype=np.int64), torch.tensor([0, 3, 1, 2])):
        ids = check_slots(slots, 4)
        assert ids.dtype == np.int32 and ids.flags.c_contiguous
        assert ids.tolist() == list(np.asarray(slots))


@pytest.mark.parametrize("slots", [[], [4], [-1], [0, 2, 0], [0, 1, 2, 3, 0], [[0, 1]], [0.0, 1.0], [True]])
def test_check_slots_refuses_bad_lists(slots):
    with pytest.raises(ValueError):
        check_slots(slots, 4)
