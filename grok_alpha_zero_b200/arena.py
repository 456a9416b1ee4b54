"""Network-vs-network matches on one GPU: is generation N+1 stronger than generation N?

`play_match` plays `n_games` games between network A and network B with the batched self-play driver
(`Self_Play.BatchedSelfPlay`): every game keeps its two PUCT trees, one per player (Self_Play.py:39-57), and the leaves of
each tree are evaluated on the device by the network of its side.  Games come in pairs that start from the same random
opening with the colours swapped, so a first-move advantage or a lucky opening counts for both networks alike.
"""
import copy
import math

import numpy as np

from . import games as G
from .Self_Play import BatchedSelfPlay, net_spec_from_configs

# random plies before the networks take over: TicTacToe is short enough to start from the empty board, Connect4 and Gomoku
# would otherwise replay the same deterministic game in every pair
DEFAULT_OPENING_PLIES = {"tictactoe": 0, "connect4": 2, "gomoku": 4}


def random_opening(game_class, plies, seed, pair):
    """Opening of pair `pair`: `plies` moves drawn uniformly among the legal moves that do not end the game, with the host
    game class and `numpy.random.Generator(PCG64([seed, pair]))`.  Returns (board int8 (H, W), next player, action ids)."""
    game = game_class()
    name = G.game_name_of(game)
    rng = np.random.Generator(np.random.PCG64([int(seed), int(pair)]))
    ids = []
    for _ in range(int(plies)):
        moves = []
        for a in game.get_legal_actions():
            g = copy.deepcopy(game)
            g.do_action(a)
            if g.check_win() == -2:
                moves.append(a)
        if not moves:
            raise ValueError("no non-terminal opening of %d plies from pair %d's position" % (plies, pair))
        a = moves[int(rng.integers(len(moves)))]
        game.do_action(a)
        ids.append(G.action_to_id(name, a))
    return np.array(game.board, dtype=np.int8), int(game.get_next_player()), ids


def elo(score):
    """Elo difference of a score in (0, 1): -400 log10(1 / score - 1); None at 0 and 1"""
    if score <= 0.0 or score >= 1.0:
        return None
    return -400.0 * math.log10(1.0 / score - 1.0)


def score_summary(scores):
    """Per-game scores of A (1 win, 0.5 draw, 0 loss) -> (score, Elo, 95 % Elo interval).  The interval maps
    score +- 1.96 sigma / sqrt(n) (sigma: standard deviation of the per-game scores) through `elo`; an end beyond 0 or 1
    becomes -inf / inf.  Elo and interval are None at score 0 or 1."""
    x = np.asarray(scores, dtype=np.float64)
    n = x.size
    s = float(x.mean())
    e = elo(s)
    if e is None:
        return s, None, None
    half = 1.96 * float(x.std()) / math.sqrt(n)
    lo, hi = elo(s - half), elo(s + half)
    return s, e, (lo if lo is not None else -math.inf, hi if hi is not None else math.inf)


def play_match(game_class, configs, weights_a, weights_b, n_games, spec_b=None, iterations=None, opening_plies=None, seed=0,
               device=0, n_slots=None):
    """Plays network A (`weights_a`, the spec that `configs` build) against network B (`weights_b`, `spec_b` or A's spec)
    on one GPU.  Sharding a match over several GPUs is not supported.

    * Pairs: games 2i and 2i+1 start from the same opening of `opening_plies` random legal, non-terminal moves
      (`random_opening(game_class, opening_plies, seed, i)`; default 0 plies for TicTacToe, 2 for Connect4, 4 for
      Gomoku).  A moves first (plays player -1) in the even games and second in the odd ones.  `n_games` must be even.
    * Move choice: by default no Dirichlet noise and tau = 0 after the opening, so a match is a deterministic function of
      (weights, seed, iterations).  `train_config["match_exploration"] = True` plays with self-play's noise
      (`dirichlet_alpha`) and tau schedule (`num_explore_actions_first/second`) instead.
    * `iterations = (ia, ib)`: iteration limits of A's and B's searches (default `int(MCTS_iteration_limit * 1.5)` for both,
      as in self-play).  `max_actions` ends a game as a draw, counting the opening's plies.
    * `n_slots`: games resident on the GPU at once (default `games_per_gpu`, 4096).

    Returns a dict: `wins` / `draws` / `losses` of A, `by_colour` (the same split by A moving first / second), `score`
    (W + D/2) / n, `elo` and its 95 % interval `elo_ci` (None at score 0 or 1), and `games`: per game `game_id`,
    `a_first`, `opening` and `actions` (action ids), `winner` (-1, 0, 1), `length` (plies, opening included) and
    `iterations` (of every search after the opening)."""
    n_games = int(n_games)
    if n_games <= 0 or n_games % 2:
        raise ValueError("n_games must be a positive even number (games come in colour-swapped pairs), got %d" % n_games)
    build_config, train_config = configs[0], configs[1]
    name = G.game_name_of(game_class())
    spec_a = net_spec_from_configs(name, build_config, train_config)
    spec_b = spec_a if spec_b is None else spec_b
    tc = dict(train_config)
    explore = bool(tc.get("match_exploration", False))
    if not explore:
        tc.update(num_explore_actions_first=0, num_explore_actions_second=0, opening_actions=False)
    if iterations is None:
        lim = int(train_config["MCTS_iteration_limit"] * 1.5)
        iterations = (lim, lim)
    plies = DEFAULT_OPENING_PLIES[name] if opening_plies is None else int(opening_plies)
    book = {}

    def opening(gid):
        pair = gid // 2
        if pair not in book:
            book[pair] = random_opening(game_class, plies, seed, pair)
        board, nxt, ids = book[pair]
        return board, nxt, ids

    slots = int(tc.get("games_per_gpu", 4096)) if n_slots is None else int(n_slots)
    sp = BatchedSelfPlay(game_class, build_config, tc, range(n_games), slots, device=device, evaluator="net", spec=spec_a,
                         weights=weights_a, seed=seed, use_noise=explore, opponent=(spec_b, weights_b), openings=opening,
                         limits=iterations)
    try:
        finished = sp.play()
    finally:
        sp.close()
    finished.sort(key=lambda g: g["game_id"])
    out = dict(wins=0, draws=0, losses=0, by_colour={"a_first": dict(wins=0, draws=0, losses=0),
                                                      "a_second": dict(wins=0, draws=0, losses=0)}, games=[])
    scores = []
    for g in finished:
        gid = g["game_id"]
        a_first = gid % 2 == 0
        a_player = -1 if a_first else 1
        w = int(g["winner"])
        res = "draws" if w == 0 else ("wins" if w == a_player else "losses")
        out[res] += 1
        out["by_colour"]["a_first" if a_first else "a_second"][res] += 1
        scores.append({"wins": 1.0, "draws": 0.5, "losses": 0.0}[res])
        opening_ids = list(book[gid // 2][2])
        actions = [int(a) for a in g["actions"]]
        out["games"].append(dict(game_id=gid, a_first=a_first, opening=opening_ids, actions=actions, winner=w,
                                 length=len(opening_ids) + len(actions), iterations=[int(i) for i in g["iterations"]]))
    out["score"], out["elo"], out["elo_ci"] = score_summary(scores)
    return out
