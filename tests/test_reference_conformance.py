"""Our game classes against outputs of the reference's own game classes and numba `*_MCTS` functions, stored under
tests/golden/ by oracle/gen_golden.py from the unmodified reference:

* kats.json.gz, random play-outs through the reference's game classes: per ply the number of legal actions, the
  action played, check_win and the input state (weighted sum every ply, in full for the first six plies);
* puct.json.gz / gumbel.json.gz, every root decision of the reference's MCTS / MCTS_Gumbel driven by the hash evaluator:
  the root's float32 priors per action, i.e. get_legal_actions_policy_MCTS applied to hash_eval(get_input_state())
  (renormalised probabilities for PUCT, masked logits for Gumbel), compared bit for bit."""
import numpy as np
import pytest

from golden_util import f32bits, load
from grok_alpha_zero_b200 import games
from hash_eval import hash_eval

OURS = {"gomoku": games.Gomoku, "connect4": games.Connect4, "tictactoe": games.TicTacToe}
KATS = load("kats.json")
ROOTS = load("puct.json") + load("gumbel.json")


def _ids(name, actions):
    return [games.action_to_id(name, a) for a in actions]


def _check_playouts(name):
    plies = 0
    for playout in KATS["games"][name]:
        g = OURS[name]()
        for p in playout:
            la = g.get_legal_actions()
            assert len(la) == p["n_legal_before"] and p["action"] in _ids(name, la)
            g.do_action(games.id_to_action(name, p["action"]))
            assert g.check_win() == p["winner"]
            st = np.asarray(g.get_input_state()).astype(np.int64).reshape(-1)
            assert int((st * np.arange(1, st.size + 1)).sum()) == p["state_sum"]
            if p["state"] is not None:
                assert st.tolist() == p["state"]
            plies += 1
    return plies


def _check_root_priors(name):
    roots = 0
    for case in (c for c in ROOTS if c["game"] == name):
        gumbel = case["mode"] == "gumbel"
        g = OURS[name]()
        for ply, mv in enumerate(case["moves"]):
            want = {r[0]: r[3] for r in mv["children"]}
            pol, _ = hash_eval(g.get_input_state(), g.policy_shape[0], gumbel, case["salt"])
            hist = np.array(g.action_history)
            acts, pri = g.get_legal_actions_policy_MCTS(g.board, -g.next_player, hist, pol.copy(), normalize=not gumbel)
            got = dict(zip(_ids(name, acts), f32bits(pri).tolist()))
            # a Gumbel root that the reference cut down to its terminal children (uniform priors over them) holds no
            # masked network output
            if not (gumbel and len(want) < len(got)):
                assert got == want, (case["mode"], case["salt"], ply)
                roots += 1
            g.do_action(games.id_to_action(name, mv["action"]))
            assert g.check_win() == mv["winner"]
    return roots


# (play-out plies, root decisions) the goldens hold per game: nothing may be left out unnoticed
CHECKED = {"tictactoe": (88, 47), "connect4": (282, 196), "gomoku": (670, 100)}


@pytest.mark.parametrize("name", ["tictactoe", "connect4", "gomoku"])
def test_static_functions_match_reference_numba(name):
    assert (_check_playouts(name), _check_root_priors(name)) == CHECKED[name]
