"""Host side of re-analysis with the production evaluators: mcts.resolve_searchers refuses evaluators that do not fit the
engines' mode, and the per-game node budgets follow muzero.evals_per_search."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from datou_gomoku_muzero_b200.mcts import host_budgets, resolve_searchers
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
])
def test_resolver_refuses(mode, evaluator):
    with pytest.raises(ValueError):
        resolve_searchers([_eng(mode), _eng(mode)], evaluator)


def test_resolver_keeps_e0_and_callables():
    assert resolve_searchers([_eng("MuZero"), _eng("AlphaZero")], "e0") == ["e0", "e0"]
    assert resolve_searchers([_eng("AlphaZero")] * 3, _ev) == [_ev] * 3


def test_host_budgets_follow_the_evaluation_schedule():
    mz = object.__new__(MuZeroDeviceSearch)          # only the engine's S and K are read
    mz.e, mz.nodes = _eng("MuZero"), 32
    rs = np.random.RandomState(0)
    boards = rs.choice(np.array([-1, 0, 1], np.int8), size=(40, 36), p=[0.4, 0.2, 0.4])
    boards[0] = 1                                     # a full board: the inactive padding root
    boards[1] = 0
    rows = host_budgets(mz, boards)
    k = np.minimum((boards == 0).sum(1), 16)
    assert rows.dtype == np.int32
    assert rows.tolist() == [evals_per_search(32, 16, int(x)) + 1 for x in k]
    assert rows[0] == 1 and rows[1] == evals_per_search(32, 16, 16) + 1
    mz.nodes = int(rows.max()) - 1
    with pytest.raises(ValueError):
        host_budgets(mz, boards)
