"""Host side of re-analysis with the production evaluators: mcts.resolve_searchers refuses evaluators that do not fit the
engines' mode, and the per-game node budgets follow muzero.evals_per_search."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from datou_gomoku_muzero_b200.mcts import E0Search, StepwiseSearch, resolve_searchers
from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, evals_per_search


def _eng(mode):
    return SimpleNamespace(mode=mode, G=4, N=6, A=36, S=32, K=16)


def _ev(obs):
    return obs, obs


@pytest.mark.parametrize("mode,evaluator", [
    ("MuZero", _ev),                                 # a callable drives the AlphaZero stepwise kernels only
    ("AlphaZero", (_ev, _ev)),                       # learned dynamics need a MuZero-mode engine
    ("MuZero", torch.nn.Linear(1, 1)),               # a module is an AlphaZero evaluator (NetworkSearch)
    ("AlphaZero", "e1"), ("MuZero", "e1"),
    ("AlphaZero", 3), ("AlphaZero", []), ("MuZero", [_ev]),
    ("AlphaZero", "e0"),                             # with logit_div=12: the fused kernels take 0 or a power of two
])
def test_resolver_refuses(mode, evaluator):
    with pytest.raises(ValueError):
        resolve_searchers([_eng(mode), _eng(mode)], evaluator, logit_div=12)


def test_resolver_wraps_e0_and_callables_in_searchers():
    engines = [_eng("MuZero"), _eng("AlphaZero")]
    got = resolve_searchers(engines, "e0", eval_seed=7, logit_div=0)
    assert len(got) == 2
    for s, e in zip(got, engines):
        assert isinstance(s, E0Search) and s.e is e and (s.seed, s.logit_div) == (7, 0)
    engines = [_eng("AlphaZero") for _ in range(3)]
    got = resolve_searchers(engines, _ev)
    assert len(got) == 3
    for s, e in zip(got, engines):
        assert isinstance(s, StepwiseSearch) and s.e is e and s.fn is _ev


def test_host_budgets_follow_the_evaluation_schedule():
    mz = object.__new__(MuZeroDeviceSearch)          # only the engine's S and K are read
    mz.e, mz.nodes = _eng("MuZero"), 32
    rs = np.random.RandomState(0)
    boards = rs.choice(np.array([-1, 0, 1], np.int8), size=(40, 36), p=[0.4, 0.2, 0.4])
    boards[0] = 1                                     # a full board: the inactive padding root
    boards[1] = 0
    rows = mz.host_budgets(boards)
    k = np.minimum((boards == 0).sum(1), 16)
    assert rows.dtype == np.int32
    assert rows.tolist() == [evals_per_search(32, 16, int(x)) + 1 for x in k]
    assert rows[0] == 1 and rows[1] == evals_per_search(32, 16, 16) + 1
    mz.nodes = int(rows.max()) - 1
    with pytest.raises(ValueError):
        mz.host_budgets(boards)
