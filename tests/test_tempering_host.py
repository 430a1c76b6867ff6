"""CPU checks of the parallel-tempering ladder rules the HMC optimizer applies before any engine exists."""
import math

import pytest

from bayesian_inference_for_nn_b200.tempering import MAX_RUNGS, geometric_ladder, validate_ladder


def test_absent_or_single_rung_means_off():
    assert validate_ladder(None) is None
    assert validate_ladder([]) is None
    assert validate_ladder([1.0]) is None
    assert validate_ladder((1,)) is None


def test_valid_ladders_come_back_as_floats():
    assert validate_ladder([1, 0.5, 0.25]) == [1.0, 0.5, 0.25]
    lad = geometric_ladder(8, 1e-3)
    assert validate_ladder(lad) == lad
    assert lad[0] == 1.0 and math.isclose(lad[-1], 1e-3)
    assert len(validate_ladder([1.0] + [0.5 ** k for k in range(1, MAX_RUNGS)])) == MAX_RUNGS


@pytest.mark.parametrize("bad", [[0.9, 0.5], [0.5], [1.0, 1.0], [1.0, 0.5, 0.7], [1.0, 0.0], [1.0, -0.1],
                                 [1.0, float("nan")], [1.0, float("inf")], [2.0, 1.0],
                                 [1.0] + [0.9 ** k for k in range(1, MAX_RUNGS + 1)], "abc", 3])
def test_invalid_ladders_are_refused(bad):
    with pytest.raises(ValueError):
        validate_ladder(bad)


@pytest.mark.parametrize("args", [(1, 0.1), (4, 0.0), (4, 1.0), (4, -1.0)])
def test_geometric_ladder_arguments(args):
    with pytest.raises(ValueError):
        geometric_ladder(*args)
