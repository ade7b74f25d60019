"""The validation schedule and best-on-validation rule of oracle/validation.py on the CPU: hand-worked schedules with
validate calls, load_state restarts and resampling schedules, and the strict-less-than rule with ties and NaN."""
import math

import numpy as np
import pytest

from oracle import validation as va


def test_every_k_steps_since_the_start():
    per_step, rows = va.schedule(3, [("run", 10)])
    assert [s for s, _, e in per_step if e] == [3, 6, 9]
    assert rows.tolist() == [3, 6, 9]


def test_chunked_runs_and_validate_calls():
    # the count runs across calls; validate adds a row at the current step without moving the schedule
    _, rows = va.schedule(4, [("validate",), ("run", 3), ("validate",), ("run", 6), ("run", 0), ("validate",)])
    assert rows.tolist() == [0, 3, 4, 8, 9]


def test_load_state_restarts_rows_and_counts_from_the_resume():
    _, rows = va.schedule(5, [("run", 7), ("load", 103), ("run", 12)])
    assert rows.tolist() == [108, 113]
    per_step, _ = va.schedule(5, [("run", 7), ("load", 103), ("run", 12)])
    assert [s for s, _, e in per_step if e] == [5, 108, 113]


@pytest.mark.parametrize("sc,freeze", [(1, va.INT64_MAX), (3, 10), (7, 4)])
def test_resampling_schedule_does_not_move_evaluations(sc, freeze):
    calls = [("run", 5), ("validate",), ("run", 9), ("load", 2), ("run", 13)]
    ref_steps, ref_rows = va.schedule(4, calls)
    steps, rows = va.schedule(4, calls, sc_sampling=sc, freeze_after=freeze)
    assert [e for _, _, e in steps] == [e for _, _, e in ref_steps]
    assert rows.tolist() == ref_rows.tolist()
    # and the resampling flags are the trainer's rule tt % sc_sampling == 0 and tt < freeze_after
    tt = [s - 1 for s, _, _ in steps]
    assert [r for _, r, _ in steps] == [t % sc == 0 and t < freeze for t in tt]


def test_best_record_strict_less_than():
    assert va.best_record([], []) == (math.inf, -1, -1)
    assert va.best_record([3.0, 2.0, 2.0, 5.0], [0, 10, 20, 30]) == (2.0, 10, 1)   # a tie keeps the earlier one
    nan = float("nan")
    assert va.best_record([nan, 4.0, nan, 1.0], [0, 1, 2, 3]) == (1.0, 3, 3)       # NaN is never taken
    b = va.best_record([nan, nan], [5, 6])
    assert b[0] == math.inf and b[1:] == (-1, -1)
    assert va.best_record([math.inf, 7.0], [1, 2]) == (7.0, 2, 1)                  # +inf is not below the start
    L = np.array([5.0, 4.0, 4.5, 1.0, 1.0, 0.5])
    assert va.best_record(L, np.arange(6) * 100) == (0.5, 500, 5)
