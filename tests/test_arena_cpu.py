"""Host side of network-vs-network matches (grok_alpha_zero_b200/arena.py): Elo arithmetic, colour assignment, openings."""
import math

import numpy as np
import pytest

from grok_alpha_zero_b200 import arena
from grok_alpha_zero_b200 import games as G
from grok_alpha_zero_b200.Self_Play import match_tree_nets


@pytest.mark.parametrize("score,want", [(0.5, 0.0), (0.75, 400 * math.log10(3)), (0.25, -400 * math.log10(3)),
                                        (10 / 11, 400.0), (0.0, None), (1.0, None)])
def test_elo_at_known_scores(score, want):
    got = arena.elo(score)
    if want is None:
        assert got is None
    else:
        assert got == pytest.approx(want, abs=1e-9)


def test_elo_interval_from_per_game_variance():
    # 3 wins, 1 loss: score 0.75, per-game standard deviation sqrt(0.75 * 0.25), 1.96 sigma / sqrt(4) around it
    s, e, (lo, hi) = arena.score_summary([1, 1, 1, 0])
    half = 1.96 * math.sqrt(0.75 * 0.25) / 2
    assert s == 0.75 and e == pytest.approx(400 * math.log10(3))
    assert lo == pytest.approx(arena.elo(0.75 - half)) and hi == math.inf    # 0.75 + half > 1
    s, e, (lo, hi) = arena.score_summary([0.5] * 10)
    assert (s, e, lo, hi) == (0.5, 0.0, 0.0, 0.0)                             # all draws: no spread
    s, e, (lo, hi) = arena.score_summary([1, 0.5, 0.5, 0] * 25)
    half = 1.96 * math.sqrt(0.125) / 10
    assert lo == pytest.approx(arena.elo(0.5 - half)) and hi == pytest.approx(-lo)
    assert arena.score_summary([1, 1]) == (1.0, None, None)
    assert arena.score_summary([0, 0, 0, 0]) == (0.0, None, None)


def test_colour_assignment():
    t = match_tree_nets(np.arange(6))
    assert t.dtype == np.uint8 and t.shape == (6, 2)
    for g in range(6):
        for k in range(2):
            assert t[g, k] == (k + g) % 2
    # tree 0 plays the first mover (-1): network 0 (A) moves first in even games, network 1 in odd ones
    assert list(t[:, 0]) == [0, 1, 0, 1, 0, 1]


@pytest.mark.parametrize("cls,plies", [(G.Connect4, 2), (G.Connect4, 9), (G.Gomoku, 4), (G.TicTacToe, 0), (G.TicTacToe, 5)])
def test_openings_are_legal_non_terminal_and_reproducible(cls, plies):
    name = G.game_name_of(cls())
    seen = set()
    for pair in range(8):
        board, nxt, ids = arena.random_opening(cls, plies, 7, pair)
        assert len(ids) == plies
        b2, n2, ids2 = arena.random_opening(cls, plies, 7, pair)   # the same for both games of a pair / on every call
        assert ids2 == ids and n2 == nxt and np.array_equal(b2, board)
        g = cls()                                                   # replay: every move legal, none ends the game
        for a in ids:
            legal = [G.action_to_id(name, x) for x in g.get_legal_actions()]
            assert a in legal
            g.do_action(G.id_to_action(name, a))
            assert g.check_win() == -2
        assert np.array_equal(np.asarray(g.board, np.int8), board) and g.get_next_player() == nxt
        seen.add(tuple(ids))
    if plies >= 2:
        assert len(seen) > 1                                        # pairs get different openings
        assert arena.random_opening(cls, plies, 8, 0)[2] != arena.random_opening(cls, plies, 7, 0)[2] or \
            arena.random_opening(cls, plies, 8, 1)[2] != arena.random_opening(cls, plies, 7, 1)[2]


def test_odd_number_of_games_is_rejected():
    build = dict(num_resnet_layers=1)
    train = dict(MCTS_iteration_limit=8, max_actions=42)
    for n in (3, 0):
        with pytest.raises(ValueError, match="even"):
            arena.play_match(G.Connect4, (build, train), None, None, n)
