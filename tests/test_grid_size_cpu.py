"""CPU: the Python surface of wva_grid_pairs_size -- a caller's status buffer must have the S*A extent."""
import numpy as np
import pytest


class _Image:
    S, A = 5, 3


@pytest.mark.parametrize("cls", ["Context", "Group"])
@pytest.mark.parametrize("bad", [np.zeros(14, dtype=np.uint8), np.zeros(15, dtype=np.int32), np.zeros((5, 3), dtype=np.uint8),
                                 np.zeros(30, dtype=np.uint8)[::2]])
def test_status_buffer_is_checked_before_the_call(wva, cls, bad):
    from inferno_autoscaler_b200 import binding
    obj = object.__new__(getattr(binding, cls))      # no device needed: the buffer is refused before the library is called
    obj.image = _Image()
    with pytest.raises(ValueError):
        obj.grid_pairs_size(bad)
