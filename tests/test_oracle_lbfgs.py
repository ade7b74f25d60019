"""CPU: the torch.optim.LBFGS driver of oracle/lbfgs.py, and the problems the device L-BFGS is tested on
(tests/test_gpu_lbfgs.py): between them every line of _strong_wolfe, _cubic_interpolate and LBFGS.step runs."""
import numpy as np
import pytest
import torch
import torch.optim.lbfgs as lb

from oracle import lbfgs as O

# lines of torch/optim/lbfgs.py that no problem runs, by their source text, with the reason
NOT_RUN = {
    'raise RuntimeError("only \'strong_wolfe\' is supported")': "line_search_fn other than None / 'strong_wolfe' is an error",
    "raise AssertionError(": "LBFGS.__init__ already refuses more than one parameter group",
    'f"Expected exactly one param_group, but got {len(self.param_groups)}"': "the message of that assertion",
}

# per problem and .step() call: (evaluations, torch's n_iter, func_evals, termination) as torch 2.11 gives them
EXPECTED = {
    "quadratic_tolerance_grad": [(23, 18, 23, 5), (1, 18, 24, 1)],
    "max_eval_in_line_search": [(7, 1, 7, 4), (6, 2, 13, 4)],
    "persisted_state_fixed_step": [(5, 5, 5, 3), (5, 10, 10, 3), (5, 15, 15, 3)],
    "fixed_step_lack_of_progress": [(2, 1, 2, 6)],
    "kink_1d": [(35, 2, 35, 6)],
}


@pytest.fixture(scope="module")
def runs():
    tr = O.CoverageTracer()
    out = {name: O.run(fg, x0, steps, free, tracer=tr, **kw) for name, (fg, x0, steps, free, kw) in O.problems().items()}
    return out, tr


def test_oracle_reproduces_a_direct_torch_run():
    fg, x0, steps, free, kw = O.problems()["persisted_state"]
    p = torch.tensor(x0, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.LBFGS([p], **kw)
    pts = []

    def closure():
        x = p.detach().numpy().copy()
        f, g = fg(x)
        pts.append(x)
        p.grad = torch.tensor(g)
        return torch.tensor(f, dtype=torch.float64)
    ends = []
    for _ in range(steps):
        opt.step(closure)
        ends.append(p.detach().numpy().copy())
    r = O.run(fg, x0, steps, free, **kw)
    assert np.array_equal(np.concatenate([q["points"] for q in r]), np.array(pts))
    for q, e in zip(r, ends):
        assert np.array_equal(q["x"], e)
    assert r[-1]["n_iter"] == opt.state[p]["n_iter"] and r[-1]["func_evals"] == opt.state[p]["func_evals"]


def test_frozen_segments_keep_their_values(runs):
    out, _ = runs
    fg, x0, steps, free, kw = O.problems()["frozen_mask"]
    x = out["frozen_mask"][-1]["x"]
    assert np.array_equal(x[500:1021], x0[500:1021])
    assert not np.array_equal(x[:500], x0[:500])


def test_problems_take_the_branches_they_are_named_for(runs):
    out, tr = runs
    for name, want in EXPECTED.items():
        got = [(q["evals"], q["n_iter"], q["func_evals"], q["reason"]) for q in out[name]]
        assert got == want, (name, got)
    # history_size 3 over more than 3 iterations keeps 3 pairs
    h3 = out["history_3"][0]
    assert h3["n_iter"] > 4 and h3["hist_len"] == 3
    # the line search runs out of evaluations: max_eval is passed as max_ls and the call stops on max_eval
    assert out["max_eval_in_line_search"][0]["reason"] == 4
    # y.s <= 1e-10 skips a pair: the test line ran more often than the line behind it
    src = open(lb.__file__).read().split("\n")
    test_line = next(k + 1 for k, s in enumerate(src) if s.strip() == "if ys > 1e-10:")
    assert tr.hits[test_line] > tr.hits[test_line + 2], "no curvature pair was skipped"
    # every termination reason (PINN_LBFGS_*) 1..7 occurs
    reasons = {q["reason"] for r in out.values() for q in r}
    assert reasons == {1, 2, 3, 4, 5, 6, 7}, reasons


def test_line_coverage_of_torch_lbfgs(runs):
    _, tr = runs
    src = open(lb.__file__).read().split("\n")
    want = O.function_lines(lb._strong_wolfe) | O.function_lines(lb._cubic_interpolate) | O.function_lines(lb.LBFGS.step)
    want = {ln for ln in want if ln <= len(src) and src[ln - 1].strip() and not src[ln - 1].strip().startswith("#")}
    missed = {ln: src[ln - 1].strip() for ln in sorted(want - tr.lines)}
    unexplained = {ln: s for ln, s in missed.items() if s not in NOT_RUN}
    assert not unexplained, unexplained
    assert len(want) > 150
