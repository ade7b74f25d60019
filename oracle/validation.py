"""The trainer's held-out validation schedule and best-on-validation rule (pinn_trainer_set_validation, include/pinn_b200.h),
restated in a few lines of numpy (TEST INFRASTRUCTURE ONLY).

A trainer with validation every `every` steps evaluates after each optimizer step that brings the steps done since the
run (re)started to a multiple of `every`, and once per pinn_trainer_validate call.  Resampling (sc_sampling,
freeze_after) decides which batch a step trains on and has no part in the schedule.  pinn_trainer_load_state(step)
restarts the rows and the record and sets the steps done to `step`.
"""
import numpy as np

INT64_MAX = (1 << 63) - 1


def schedule(every, calls, step0=0, sc_sampling=1, freeze_after=INT64_MAX):
    """calls: the trainer calls in order, ("run", k) | ("validate",) | ("load", step), on a trainer created with
    step0 steps done.  -> list of (steps done after the step, resampled, evaluated) per optimizer step, and the steps-done
    column of the rows read_validation returns (the rows since the last load)."""
    steps, base, per_step, rows = step0, step0, [], []
    for c in calls:
        if c[0] == "run":
            for _ in range(int(c[1])):
                resampled = steps % sc_sampling == 0 and steps < freeze_after
                steps += 1
                evaluated = (steps - base) % every == 0
                per_step.append((steps, resampled, evaluated))
                if evaluated:
                    rows.append(steps)
        elif c[0] == "validate":
            rows.append(steps)
        elif c[0] == "load":
            steps = base = int(c[1])
            rows = []
        else:
            raise ValueError("unknown call %r" % (c,))
    return per_step, np.asarray(rows, np.int64)


def best_record(losses, steps):
    """The best-on-validation record over evaluations in order: it starts at +inf / step -1 and takes an evaluation only
    when its loss is strictly lower, so a tie keeps the earlier one and a NaN is never taken.
    -> (best loss, its step, its index or -1)."""
    best, step, idx = np.inf, -1, -1
    for i, (L, s) in enumerate(zip(losses, steps)):
        if L < best:
            best, step, idx = float(L), int(s), i
    return best, step, idx
