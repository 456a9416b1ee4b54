"""Network-vs-network matches and tournaments on one GPU: is generation N+1 stronger than generation N, and where does
every generation stand?

`play_match` plays `n_games` games between network A and network B with the batched self-play driver
(`Self_Play.BatchedSelfPlay`): every game keeps its two PUCT trees, one per player (Self_Play.py:39-57), and the leaves of
each tree are evaluated on the device by the network of its side.  Games come in pairs that start from the same random
opening with the colours swapped, so a first-move advantage or a lucky opening counts for both networks alike.

`play_tournament` plays a schedule of such matches between 2..8 networks (a round robin or a gauntlet) in ONE batch on the
device, each pair's games exactly as `play_match` would play them, and fits one Bradley-Terry Elo ladder to the crosstable.
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


def opening_book(game_class, plies, seed):
    """opening(pair) -> random_opening(game_class, plies, seed, pair), each pair's opening drawn once"""
    book = {}

    def opening(pair):
        if pair not in book:
            book[pair] = random_opening(game_class, plies, seed, pair)
        return book[pair]
    return opening


def _match_config(game_class, configs, n_nets, iterations, opening_plies, symmetry):
    """(game name, build config, train config of the match, exploration on?, per-network iteration limits, opening plies)"""
    build_config, train_config = configs[0], configs[1]
    name = G.game_name_of(game_class())
    tc = dict(train_config, eval_symmetry=symmetry)
    explore = bool(tc.get("match_exploration", False))
    if not explore:
        tc.update(num_explore_actions_first=0, num_explore_actions_second=0, opening_actions=False)
    if iterations is None:
        iterations = (int(train_config["MCTS_iteration_limit"] * 1.5),) * n_nets
    if len(iterations) != n_nets:
        raise ValueError("iterations: %d limits for %d networks" % (len(iterations), n_nets))
    plies = DEFAULT_OPENING_PLIES[name] if opening_plies is None else int(opening_plies)
    return name, build_config, tc, explore, tuple(int(x) for x in iterations), plies


def _outcome(winner, first):
    """'wins' / 'draws' / 'losses' of the network that played player -1 (first) or player 1"""
    if winner == 0:
        return "draws"
    return "wins" if winner == (-1 if first else 1) else "losses"


def tally(outcomes, colour_keys=("a_first", "a_second")):
    """[(moved first?, 'wins' | 'draws' | 'losses'), ...] of one side -> wins / draws / losses, by_colour (split by
    colour_keys), score, elo, elo_ci (score_summary)"""
    out = dict(wins=0, draws=0, losses=0, by_colour={k: dict(wins=0, draws=0, losses=0) for k in colour_keys})
    scores = []
    for first, res in outcomes:
        out[res] += 1
        out["by_colour"][colour_keys[0] if first else colour_keys[1]][res] += 1
        scores.append({"wins": 1.0, "draws": 0.5, "losses": 0.0}[res])
    out["score"], out["elo"], out["elo_ci"] = score_summary(scores)
    return out


def play_match(game_class, configs, weights_a, weights_b, n_games, spec_b=None, iterations=None, opening_plies=None, seed=0,
               device=0, n_slots=None, symmetry="none"):
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
    * `symmetry`: how both networks evaluate a position (Engine.set_eval_symmetry): "none" (default, once as reached, the
      reference's evaluation), "random" (one hashed board symmetry per request) or "ensemble" (the mean over all board
      symmetries: a stronger, lower-variance evaluator at n times the network work - 8 for Gomoku / TicTacToe, 2 for
      Connect4).  Only "none" keeps reference parity.

    Returns a dict: `wins` / `draws` / `losses` of A, `by_colour` (the same split by A moving first / second), `score`
    (W + D/2) / n, `elo` and its 95 % interval `elo_ci` (None at score 0 or 1), and `games`: per game `game_id`,
    `a_first`, `opening` and `actions` (action ids), `winner` (-1, 0, 1), `length` (plies, opening included) and
    `iterations` (of every search after the opening)."""
    n_games = int(n_games)
    if n_games <= 0 or n_games % 2:
        raise ValueError("n_games must be a positive even number (games come in colour-swapped pairs), got %d" % n_games)
    name, build_config, tc, explore, iterations, plies = _match_config(game_class, configs, 2, iterations, opening_plies, symmetry)
    spec_a = net_spec_from_configs(name, build_config, configs[1])
    spec_b = spec_a if spec_b is None else spec_b
    book = opening_book(game_class, plies, seed)

    def opening(gid):
        return book(gid // 2)

    slots = int(tc.get("games_per_gpu", 4096)) if n_slots is None else int(n_slots)
    sp = BatchedSelfPlay(game_class, build_config, tc, range(n_games), slots, device=device, evaluator="net", spec=spec_a,
                         weights=weights_a, seed=seed, use_noise=explore, opponent=(spec_b, weights_b), openings=opening,
                         limits=iterations)
    try:
        finished = sp.play()
    finally:
        sp.close()
    finished.sort(key=lambda g: g["game_id"])
    games = []
    for g in finished:
        gid = g["game_id"]
        opening_ids = list(book(gid // 2)[2])
        actions = [int(a) for a in g["actions"]]
        games.append(dict(game_id=gid, a_first=gid % 2 == 0, opening=opening_ids, actions=actions, winner=int(g["winner"]),
                          length=len(opening_ids) + len(actions), iterations=[int(i) for i in g["iterations"]]))
    out = tally([(g["a_first"], _outcome(g["winner"], g["a_first"])) for g in games])
    out["games"] = games
    return out


# ------------------------------------------------------------------------------------------------ tournaments --
MAX_NETS = 8   # GAZ_MAX_NETS: networks one engine can hold


def round_robin(n_nets):
    """every pair once: (i, j) for i < j, in lexicographic order"""
    return [(i, j) for i in range(n_nets) for j in range(i + 1, n_nets)]


def gauntlet(n_nets):
    """network 0 against each of the others: (0, j) for j = 1..n_nets-1"""
    return [(0, j) for j in range(1, n_nets)]


def check_schedule(n_nets, games_per_pair, pairs):
    """validated schedule: list of (i, j) with i != j, both < n_nets; 2 <= n_nets <= 8; games_per_pair even"""
    if not 2 <= n_nets <= MAX_NETS:
        raise ValueError("a tournament needs 2 to %d networks, got %d" % (MAX_NETS, n_nets))
    if games_per_pair <= 0 or games_per_pair % 2:
        raise ValueError("games_per_pair must be a positive even number (games come in colour-swapped pairs), got %d"
                         % games_per_pair)
    pairs = round_robin(n_nets) if pairs is None else [(int(i), int(j)) for i, j in pairs]
    if not pairs:
        raise ValueError("the schedule has no pair")
    for i, j in pairs:
        if i == j:
            raise ValueError("pair (%d, %d): a network cannot play itself" % (i, j))
        if not (0 <= i < n_nets and 0 <= j < n_nets):
            raise ValueError("pair (%d, %d): network index out of range 0..%d" % (i, j, n_nets - 1))
    return pairs


def tournament_game(game_id, pairs, games_per_pair):
    """global game id -> (pair index p, local id l within the pair, network moving first, network moving second).  Pair p
    owns ids [p * G, (p + 1) * G); as in play_match, i of pair (i, j) moves first (plays player -1) in the even local games."""
    p, l = divmod(int(game_id), int(games_per_pair))
    i, j = pairs[p]
    return (p, l, i, j) if l % 2 == 0 else (p, l, j, i)


def tournament_tree_nets(pairs, games_per_pair):
    """tree_nets(game_id) -> (network of tree 0, network of tree 1) for BatchedSelfPlay.  Tree 0 plays player -1, so it
    belongs to the network moving first."""
    def tree_nets(game_id):
        _, _, first, second = tournament_game(game_id, pairs, games_per_pair)
        return first, second
    return tree_nets


ELO_PER_NAT = 400.0 / math.log(10.0)


def _strongly_connected(beat):
    """is the digraph of the boolean adjacency matrix `beat` strongly connected?"""
    n = beat.shape[0]

    def reach(adj):
        seen = np.zeros(n, bool)
        seen[0] = True
        stack = [0]
        while stack:
            u = stack.pop()
            for v in np.nonzero(adj[u] & ~seen)[0]:
                seen[v] = True
                stack.append(int(v))
        return seen.all()
    return reach(beat) and reach(beat.T)


def bradley_terry(points, games):
    """Maximum-likelihood Bradley-Terry ratings from a crosstable.  points[i][j]: what i scored against j (a win 1, a draw
    1/2 to each side); games[i][j] = games[j][i]: games between them.  P(i beats j) = 1 / (1 + 10^((r_j - r_i) / 400)).

    Returns (ratings, None) with ratings = dict(elo, elo_ci, se): Elo per network with network 0 at 0, the standard
    errors and 95 % intervals from the inverse Fisher information with network 0's row and column removed (network 0:
    0, (0, 0)).  Fitted by Newton's method on the concave log-likelihood.  When the digraph "i scored against j" is not
    strongly connected the maximum does not exist (some rating runs off to infinity): returns (None, reason)."""
    S = np.asarray(points, np.float64)
    N = np.asarray(games, np.float64)
    K = S.shape[0]
    if S.shape != (K, K) or N.shape != (K, K) or not np.allclose(N, N.T) or not np.allclose(S + S.T, N):
        raise ValueError("points / games: K x K, games symmetric, points[i][j] + points[j][i] == games[i][j]")
    idle = [k for k in range(K) if N[k].sum() == 0]
    if idle:
        return None, "network(s) %s played no games: their ratings are undetermined" % idle
    if not _strongly_connected(S > 0):
        return None, ("the results are not strongly connected (some network or group of networks scored nothing against "
                      "the rest), so the maximum-likelihood ratings do not exist")
    theta = np.zeros(K)

    def loglik(t):
        d = t[:, None] - t[None, :]
        return float((S * -np.logaddexp(0.0, -d)).sum())

    def grad_hess(t):
        p = 1.0 / (1.0 + np.exp(t[None, :] - t[:, None]))   # p[i, j] = P(i beats j)
        g = S.sum(1) - (N * p).sum(1)
        w = N * p * p.T
        H = w - np.diag(w.sum(1))
        return g, H

    ll = loglik(theta)
    for _ in range(200):
        g, H = grad_hess(theta)
        step = np.zeros(K)
        step[1:] = np.linalg.solve(-H[1:, 1:], g[1:])
        t = 1.0
        while t > 1e-8:               # damped Newton: the log-likelihood never decreases
            cand = theta + t * step
            cl = loglik(cand)
            if cl >= ll - 1e-12 * abs(ll):
                break
            t *= 0.5
        theta, ll = cand, cl
        if np.abs(t * step).max() < 1e-13:
            break
    _, H = grad_hess(theta)
    cov = np.linalg.inv(-H[1:, 1:])
    se = np.concatenate([[0.0], np.sqrt(np.diag(cov))]) * ELO_PER_NAT
    elo_r = theta * ELO_PER_NAT
    ci = [(float(r - 1.96 * e), float(r + 1.96 * e)) for r, e in zip(elo_r, se)]
    return dict(elo=[float(x) for x in elo_r], se=[float(x) for x in se], elo_ci=ci), None


def play_tournament(game_class, configs, weights, games_per_pair, specs=None, pairs=None, iterations=None,
                    opening_plies=None, seed=0, device=0, n_slots=None, symmetry="none"):
    """Plays a tournament of K = len(weights) networks (2..8) on one GPU, every scheduled pair's games in one batch.

    * `pairs`: the schedule, by default the round robin (i, j), i < j (`round_robin`); a gauntlet is `gauntlet(K)`.
    * Pair p plays `games_per_pair` (even) games with global ids [p * G, (p + 1) * G).  Within the pair, i takes A's role
      of play_match: i moves first in the even local games, and local game l starts from
      `random_opening(game_class, opening_plies, seed, l // 2)`.  So every pair meets the same opening suite, and each
      pair's games equal `play_match(weights[i], weights[j], G, seed=seed)` game for game (with the deterministic
      defaults: no noise, tau = 0; `train_config["match_exploration"]` plays with noise as play_match does).
    * `specs`: the K network specs (default: every network has the spec that `configs` build).  Networks of equal specs
      share one activation workspace on the device.
    * `iterations`: the K per-network iteration limits (default `int(MCTS_iteration_limit * 1.5)` for each).
    * `n_slots`: games resident on the GPU at once (default `games_per_gpu`, 4096); finished games are replaced by the
      next ones in id order, so pairs mix in the batch.
    * `symmetry`: "none" (default, reference parity), "random" or "ensemble", for every network (as play_match).

    Returns a dict:
    * `pairs`: per scheduled pair `i`, `j`, wins / draws / losses of i, `by_colour` (i_first / i_second), `score` of i,
      `elo` and `elo_ci` (as play_match);
    * `crosstable`: K x K, [i][j] = i's score against j over all their games; NaN where no games were played;
    * `ratings`: Bradley-Terry Elo of every network (`bradley_terry`: network 0 at 0, `se`, 95 % `elo_ci`), or None with
      the reason in `ratings_reason`;
    * `games`: per game `game_id`, `pair`, `first`, `second` (network indices), `opening`, `actions`, `winner`, `length`,
      `iterations` (as play_match)."""
    K = len(weights)
    G_ = int(games_per_pair)
    pairs = check_schedule(K, G_, pairs)
    name, build_config, tc, explore, iterations, plies = _match_config(game_class, configs, K, iterations, opening_plies, symmetry)
    default_spec = net_spec_from_configs(name, build_config, configs[1])
    specs = [default_spec] * K if specs is None else [default_spec if s is None else s for s in specs]
    if len(specs) != K:
        raise ValueError("specs: %d specs for %d networks" % (len(specs), K))
    book = opening_book(game_class, plies, seed)

    def opening(gid):
        return book(tournament_game(gid, pairs, G_)[1] // 2)

    n_games = len(pairs) * G_
    slots = int(tc.get("games_per_gpu", 4096)) if n_slots is None else int(n_slots)
    sp = BatchedSelfPlay(game_class, build_config, tc, range(n_games), slots, device=device, evaluator="net", spec=specs[0],
                         weights=weights[0], seed=seed, use_noise=explore,
                         opponents=[(specs[k], weights[k]) for k in range(1, K)],
                         tree_nets=tournament_tree_nets(pairs, G_), openings=opening, limits=iterations)
    try:
        finished = sp.play()
    finally:
        sp.close()
    finished.sort(key=lambda g: g["game_id"])
    games = []
    for g in finished:
        gid = g["game_id"]
        p, l, first, second = tournament_game(gid, pairs, G_)
        opening_ids = list(book(l // 2)[2])
        actions = [int(a) for a in g["actions"]]
        games.append(dict(game_id=gid, pair=p, first=first, second=second, opening=opening_ids, actions=actions,
                          winner=int(g["winner"]), length=len(opening_ids) + len(actions),
                          iterations=[int(i) for i in g["iterations"]]))
    points = np.zeros((K, K))
    count = np.zeros((K, K))
    out_pairs = []
    for p, (i, j) in enumerate(pairs):
        outcomes = [(g["first"] == i, _outcome(g["winner"], g["first"] == i)) for g in games if g["pair"] == p]
        t = tally(outcomes, ("i_first", "i_second"))
        out_pairs.append(dict(i=i, j=j, **t))
        pts = t["wins"] + 0.5 * t["draws"]
        points[i, j] += pts
        points[j, i] += len(outcomes) - pts
        count[i, j] += len(outcomes)
        count[j, i] += len(outcomes)
    with np.errstate(invalid="ignore", divide="ignore"):
        cross = np.where(count > 0, points / np.where(count > 0, count, 1), np.nan)
    ratings, reason = bradley_terry(points, count)
    return dict(pairs=out_pairs, crosstable=cross.tolist(), ratings=ratings, ratings_reason=reason, games=games)
