"""Host side of tournaments (arena.py): the Bradley-Terry fit, the schedule and its game-id mapping."""
import math

import numpy as np
import pytest

from grok_alpha_zero_b200 import arena
from grok_alpha_zero_b200 import games as G


def _table(K, results):
    """results: {(i, j): (wins of i, draws, losses of i)} -> (points, games)"""
    S, N = np.zeros((K, K)), np.zeros((K, K))
    for (i, j), (w, d, l) in results.items():
        S[i, j] += w + 0.5 * d
        S[j, i] += l + 0.5 * d
        N[i, j] += w + d + l
        N[j, i] += w + d + l
    return S, N


@pytest.mark.parametrize("w,d,l", [(7, 2, 3), (1, 0, 9), (40, 13, 11), (5, 5, 5)])
def test_two_players_rate_like_elo_of_the_score(w, d, l):
    S, N = _table(2, {(0, 1): (w, d, l)})
    r, why = arena.bradley_terry(S, N)
    assert why is None
    score_1 = (l + 0.5 * d) / (w + d + l)
    assert r["elo"][0] == 0.0
    assert abs(r["elo"][1] - arena.elo(score_1)) < 1e-9


def test_symmetric_crosstable_rates_everyone_zero():
    S, N = _table(4, {(i, j): (3, 2, 3) for i in range(4) for j in range(i + 1, 4)})
    r, why = arena.bradley_terry(S, N)
    assert why is None
    np.testing.assert_allclose(r["elo"], 0.0, atol=1e-9)
    assert r["se"][0] == 0.0 and all(x > 0 for x in r["se"][1:])


def test_recovers_known_ratings_inside_the_intervals():
    truth = np.array([0.0, 120.0, -80.0, 250.0, 30.0])
    rng = np.random.default_rng(7)
    res = {}
    for i in range(5):
        for j in range(i + 1, 5):
            p = 1.0 / (1.0 + 10.0 ** ((truth[j] - truth[i]) / 400.0))
            w = int(rng.binomial(4000, p))
            res[(i, j)] = (w, 0, 4000 - w)
    r, why = arena.bradley_terry(*_table(5, res))
    assert why is None
    for k in range(1, 5):
        lo, hi = r["elo_ci"][k]
        assert lo <= truth[k] <= hi, (k, r["elo"][k], (lo, hi), truth[k])
        assert hi - lo < 60.0


def test_four_times_the_games_halves_the_standard_errors():
    S, N = _table(3, {(0, 1): (5, 2, 3), (0, 2): (2, 1, 7), (1, 2): (4, 4, 2)})
    r1, _ = arena.bradley_terry(S, N)
    r4, _ = arena.bradley_terry(4 * S, 4 * N)
    np.testing.assert_allclose(r4["elo"], r1["elo"], atol=1e-9)
    np.testing.assert_allclose(np.array(r4["se"][1:]) * 2.0, r1["se"][1:], rtol=1e-9)


def test_not_strongly_connected_has_no_ratings():
    # network 2 won every game it played: no finite maximum-likelihood rating
    S, N = _table(3, {(0, 1): (3, 1, 2), (2, 0): (4, 0, 0), (2, 1): (4, 0, 0)})
    r, why = arena.bradley_terry(S, N)
    assert r is None and "strongly connected" in why
    # a network that played nobody
    S, N = _table(3, {(0, 1): (3, 1, 2)})
    r, why = arena.bradley_terry(S, N)
    assert r is None and "no games" in why


def test_round_robin_and_gauntlet_order():
    assert arena.round_robin(4) == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    assert len(arena.round_robin(8)) == 28
    assert arena.gauntlet(4) == [(0, 1), (0, 2), (0, 3)]
    assert arena.check_schedule(3, 4, None) == arena.round_robin(3)


def test_game_id_mapping():
    pairs = arena.round_robin(3)        # (0,1) (0,2) (1,2)
    G_ = 6
    got = [arena.tournament_game(g, pairs, G_) for g in range(len(pairs) * G_)]
    for gid, (p, l, first, second) in enumerate(got):
        assert p == gid // G_ and l == gid % G_
        i, j = pairs[p]
        assert (first, second) == ((i, j) if l % 2 == 0 else (j, i))
    assert got[7] == (1, 1, 2, 0)


def test_tree_nets_colours():
    """tree 0 plays player -1 (moves first): it belongs to the first network; pair (i, j) of a 2-network tournament is
    exactly the match colouring (Self_Play.match_tree_nets)"""
    from grok_alpha_zero_b200.Self_Play import match_tree_nets
    tn = arena.tournament_tree_nets([(0, 1)], 8)
    np.testing.assert_array_equal(np.array([tn(g) for g in range(8)]), match_tree_nets(range(8)))
    tn = arena.tournament_tree_nets([(2, 5), (4, 1)], 4)
    assert [tn(g) for g in range(8)] == [(2, 5), (5, 2), (2, 5), (5, 2), (4, 1), (1, 4), (4, 1), (1, 4)]


@pytest.mark.parametrize("K,G_,pairs,msg", [
    (3, 5, None, "even"),
    (3, 0, None, "even"),
    (3, 4, [(1, 1)], "itself"),
    (3, 4, [(0, 3)], "out of range"),
    (3, 4, [(-1, 2)], "out of range"),
    (1, 4, None, "2 to 8"),
    (9, 4, None, "2 to 8"),
])
def test_schedule_rejections(K, G_, pairs, msg):
    with pytest.raises(ValueError, match=msg):
        arena.check_schedule(K, G_, pairs)


def test_play_tournament_rejects_before_touching_the_device():
    cfg = ({"use_stablemax": False}, dict(MCTS_iteration_limit=10, max_actions=42))
    for weights, G_ in (([{}] * 3, 3), ([{}], 2), ([{}] * 9, 2)):
        with pytest.raises(ValueError):
            arena.play_tournament(G.Connect4, cfg, weights, G_)
    with pytest.raises(ValueError, match="iterations"):
        arena.play_tournament(G.Connect4, cfg, [{}] * 3, 2, iterations=(10, 10))
    assert math.isfinite(arena.ELO_PER_NAT)
