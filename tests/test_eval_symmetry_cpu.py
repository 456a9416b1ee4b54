"""Host side of symmetric network evaluation: the symmetry tables of games.eval_symmetries and the Python twin of the
device's GAZ_SYM_RANDOM hash (oracle/sym_hash.py)."""
import numpy as np
import pytest

import sym_hash
from grok_alpha_zero_b200 import games as G
from grok_alpha_zero_b200.engine import DIMS

CLASSES = {"gomoku": G.Gomoku, "connect4": G.Connect4, "tictactoe": G.TicTacToe}
GAMES = ["gomoku", "connect4", "tictactoe"]


def _ids(name, actions):
    return {G.action_to_id(name, a) for a in actions}


def random_game(name, rng, plies):
    """a game of `plies` random legal moves (fewer if the board fills up); returns (game, action ids)"""
    g = CLASSES[name]()
    ids = []
    for _ in range(plies):
        legal = sorted(_ids(name, g.get_legal_actions()))
        if not legal:
            break
        a = legal[rng.randint(len(legal))]
        g.do_action(G.id_to_action(name, a))
        ids.append(a)
    return g, ids


@pytest.mark.parametrize("name", GAMES)
def test_rows_are_permutations_and_row_0_is_the_identity(name):
    H, W, C, P = DIMS[name]
    ps, pp = G.eval_symmetries(name)
    n = 2 if name == "connect4" else 8
    assert ps.shape == (n, H * W * C) and pp.shape == (n, P)
    assert ps.dtype == np.int32 and pp.dtype == np.int32
    for tab, size in ((ps, H * W * C), (pp, P)):
        for row in tab:
            np.testing.assert_array_equal(np.sort(row), np.arange(size))
        np.testing.assert_array_equal(tab[0], np.arange(size))
    assert len({r.tobytes() for r in ps}) == n and len({r.tobytes() for r in pp}) == n


@pytest.mark.parametrize("name", GAMES)
def test_the_set_is_closed_under_composition(name):
    ps, pp = G.eval_symmetries(name)
    for tab in (ps, pp):
        rows = {r.tobytes() for r in tab}
        for a in tab:
            for b in tab:
                assert a[b].tobytes() in rows


@pytest.mark.parametrize("name", GAMES)
def test_transformed_games_replay_to_the_gathered_state(name):
    """For every g: replaying the actions mapped through perm_policy[g] gives the state gathered through perm_state[g],
    and the legal actions map through perm_policy[g]."""
    ps, pp = G.eval_symmetries(name)
    P = DIMS[name][3]
    rng = np.random.RandomState(7)
    max_plies = {"gomoku": 40, "connect4": 30, "tictactoe": 8}[name]
    for trial in range(12):
        game, ids = random_game(name, rng, rng.randint(0, max_plies + 1))
        state = np.asarray(game.get_input_state()).reshape(-1)
        legal = np.zeros(P, bool)
        legal[list(_ids(name, game.get_legal_actions()))] = True
        for g in range(len(ps)):
            t = CLASSES[name]()
            for a in ids:
                t.do_action(G.id_to_action(name, int(pp[g][a])))
            np.testing.assert_array_equal(np.asarray(t.get_input_state()).reshape(-1), state[ps[g]], err_msg="g=%d" % g)
            legal_t = np.zeros(P, bool)
            legal_t[list(_ids(name, t.get_legal_actions()))] = True
            np.testing.assert_array_equal(legal_t[pp[g]], legal)


def test_connect4_uses_the_column_mirror_not_the_augmentation_row_flip():
    ps, pp = G.eval_symmetries("connect4")
    np.testing.assert_array_equal(pp[1], np.arange(7)[::-1])
    game, _ = random_game("connect4", np.random.RandomState(3), 9)
    st = np.asarray(game.get_input_state())                      # (6, 7, 4)
    mirrored = st.reshape(-1)[ps[1]].reshape(6, 7, 4)
    np.testing.assert_array_equal(mirrored, st[:, ::-1, :])
    aug, _ = G.Connect4.augment_sample(st[None], np.zeros((1, 7), np.float32))
    assert not np.array_equal(mirrored, aug[1][0])               # augment_sample flips the rows (a reference quirk)
    np.testing.assert_array_equal(aug[1][0], st[::-1])


def test_symmetry_hash_twin_is_deterministic_and_reaches_every_g():
    rng = np.random.RandomState(0)
    for name, n in (("gomoku", 8), ("connect4", 2), ("tictactoe", 8)):
        draws = []
        for i in range(120):
            game, _ = random_game(name, rng, rng.randint(0, 9))
            st = game.get_input_state()
            key = sym_hash.tree_key(11, i)
            g = sym_hash.sym_draw(st, 11, key, n)
            assert 0 <= g < n and g == sym_hash.sym_draw(np.array(st, copy=True), 11, key, n)
            draws.append(g)
        assert set(draws) == set(range(n)), (name, draws)
    st = np.zeros((15, 15, 2), np.int8)
    assert len({sym_hash.sym_draw(st, s, 5, 8) for s in range(64)}) == 8          # the seed changes the draw
    assert len({sym_hash.sym_draw(st, 3, k, 8) for k in range(64)}) == 8          # so does the tree key
    assert sym_hash.tree_key(5, 3) == 6 and sym_hash.tree_key(5, 3, np.array([9, 9, 9, 42], np.uint64)) == 42
