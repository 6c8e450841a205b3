"""CPU: the Python surface of wva_analyze_scenarios -- the scenario rates must be a finite float32 [n_scen, S] array with
1 <= n_scen <= 1024; anything else is refused before the library is called."""
import numpy as np
import pytest


class _Image:
    S, A, T = 5, 3, 2


_BAD = [
    ("list", [[1.0] * 5]),
    ("float64", np.ones((2, 5), dtype=np.float64)),
    ("int32", np.ones((2, 5), dtype=np.int32)),
    ("1-d", np.ones(5, dtype=np.float32)),
    ("3-d", np.ones((1, 2, 5), dtype=np.float32)),
    ("wrong S", np.ones((2, 4), dtype=np.float32)),
    ("no scenario", np.ones((0, 5), dtype=np.float32)),
    ("1025 scenarios", np.ones((1025, 5), dtype=np.float32)),
    ("nan", np.array([[1.0, np.nan, 1.0, 1.0, 1.0]], dtype=np.float32)),
    ("inf", np.array([[1.0, 1.0, np.inf, 1.0, 1.0]], dtype=np.float32)),
    ("-inf", np.array([[1.0, 1.0, 1.0, 1.0, -np.inf]], dtype=np.float32)),
]


@pytest.mark.parametrize("cls", ["Context", "Group"])
@pytest.mark.parametrize("name,bad", _BAD, ids=[n for n, _ in _BAD])
def test_scenario_rates_are_checked_before_the_call(wva, cls, name, bad):
    from inferno_autoscaler_b200 import binding
    obj = object.__new__(getattr(binding, cls))      # no device needed: the rates are refused before the library is called
    obj.image = _Image()
    with pytest.raises((TypeError, ValueError)):
        obj.analyze_scenarios(bad)


def test_accepted_rates_are_contiguous_float32():
    from inferno_autoscaler_b200 import binding
    r = np.arange(20, dtype=np.float32).reshape(5, 4).T            # a transposed view: (4, 5), not C-contiguous
    out = binding._scenario_rates(r, 5)
    assert out.flags.c_contiguous and out.dtype == np.float32 and np.array_equal(out, r)
    neg = -np.ones((1024, 5), dtype=np.float32)                    # negative rates are valid input (nil allocations)
    assert binding._scenario_rates(neg, 5) is neg
