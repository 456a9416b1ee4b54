"""GPU suite: two networks attached to one engine (gaz_attach_nets / gaz_set_tree_nets) and the match driver (arena.py)."""
import numpy as np
import pytest

import engine_parity as ep
import oracle as orc
from grok_alpha_zero_b200 import arena, netspec
from grok_alpha_zero_b200 import games as G
from grok_alpha_zero_b200.Self_Play import BatchedSelfPlay, net_spec_from_configs
from grok_alpha_zero_b200.engine import Engine, EngineError
from grok_alpha_zero_b200.net import Net

pytestmark = pytest.mark.gpu

SPECS = {"tictactoe": {}, "connect4": dict(num_blocks=2), "gomoku": dict(num_blocks=2, use_se=True)}
CLASSES = {"tictactoe": G.TicTacToe, "connect4": G.Connect4, "gomoku": G.Gomoku}


def spec_of(game):
    return netspec.build_spec(game, "softmax", **SPECS[game])


def search(game, nets, tree_net, n_games, iters, seed=0):
    """n_games random positions, one tree each, searched to `iters` with graph-replayed rounds; nets = [A] attaches A
    alone, [A, B] attaches both and maps tree t to nets[tree_net[t]].  Returns root_dense (visits, value sums, info)."""
    eng = Engine(game, n_games=n_games, mode="puct", trees_per_game=1, c_puct_init=2.5, iters_hint=iters)
    if len(nets) == 1:
        nets[0].attach(eng)
    else:
        eng.attach_nets(nets)
        eng.set_tree_nets(tree_net)
    rng = np.random.RandomState(seed)
    for i in range(n_games):
        g = ep.random_position(game, rng, rng.randint(0, 6))
        eng.set_game(i, g.board, g.next_player, g.history)
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([iters] * n_games)
    while eng.remaining() > 0:
        eng.rounds_net(16)
    assert eng.status() == 0
    out = eng.root_dense()
    eng.close()
    return out


@pytest.mark.parametrize("game", ["tictactoe", "connect4", "gomoku"])
def test_routing_is_invisible_when_both_networks_are_the_same(game):
    """Rows of a forward pass are bit-independent of their position in the batch, so routing every tree's leaves through
    a second network with the same weights must change no bit of the search, whatever the mapping."""
    spec = spec_of(game)
    W = netspec.init_weights(spec, seed=3)
    n_games, iters = 40, 60
    a, a2 = Net(spec, W, max_batch=16), Net(spec, W, max_batch=16)   # 40 trees: three chunks per network
    ref = search(game, [a], None, n_games, iters)
    one = np.zeros(n_games, np.uint8)
    one[17] = 1
    for mapping in (np.random.RandomState(1).randint(0, 2, n_games), np.ones(n_games), one):
        got = search(game, [a, a2], mapping, n_games, iters)
        np.testing.assert_array_equal(got[0], ref[0])
        np.testing.assert_array_equal(got[1].view(np.uint32), ref[1].view(np.uint32))
        np.testing.assert_array_equal(got[2], ref[2])
    a.close(); a2.close()


@pytest.mark.parametrize("game,iters", [("connect4", 120), ("gomoku", 150)])
def test_each_tree_searches_with_its_own_network(game, iters):
    """Two networks with different weights and a random mapping: every tree's root statistics equal the C oracle's
    search with the host forward of that tree's network as its evaluator."""
    spec = spec_of(game)
    nets = [Net(spec, netspec.init_weights(spec, seed=2), max_batch=4), Net(spec, netspec.init_weights(spec, seed=5), max_batch=4)]
    n_games = 10
    mapping = np.random.RandomState(4).randint(0, 2, n_games).astype(np.uint8)
    mapping[:2] = [0, 1]
    eng = Engine(game, n_games=n_games, mode="puct", trees_per_game=1, c_puct_init=2.5, iters_hint=iters)
    eng.attach_nets(nets)
    eng.set_tree_nets(mapping)
    rng = np.random.RandomState(0)
    games = [ep.random_position(game, rng, rng.randint(0, 8)) for _ in range(n_games)]
    for i, g in enumerate(games):
        eng.set_game(i, g.board, g.next_player, g.history)
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([iters] * n_games)
    while eng.remaining() > 0:
        eng.rounds_net(16)
    assert eng.status() == 0
    for i, g in enumerate(games):
        net = nets[mapping[i]]

        def host_eval(state, net=net):
            p, v = net.forward(state[None])
            return p[0], v[0]

        t = orc.OracleTree(game, False, evaluator=host_eval, c_puct_init=2.5)
        t.new_root(g)
        t.run(iters)
        ref = t.root_stats()
        st = eng.root_stats(i)
        np.testing.assert_array_equal(st["action"], ref["action"])
        np.testing.assert_array_equal(st["visits"], ref["visits"])
        np.testing.assert_array_equal(st["values"].view(np.uint32), ref["values"].view(np.uint32))
    eng.close()
    for n in nets:
        n.close()


def test_the_mapping_survives_graph_replay():
    """set_tree_nets after the round graph was captured: the replayed graph reads the new table (run A) exactly as eager
    rounds do (run B, Net.profile on); run C keeps the first mapping and must differ."""
    spec = spec_of("connect4")
    Wa, Wb = netspec.init_weights(spec, seed=2), netspec.init_weights(spec, seed=6)
    m1 = np.array([0, 1] * 4, np.uint8)
    m2 = 1 - m1

    def run(graph, switch):
        nets = [Net(spec, Wa, max_batch=4), Net(spec, Wb, max_batch=4)]
        if not graph:
            for n in nets:
                n.profile(8192)
        eng = Engine("connect4", n_games=8, mode="puct", trees_per_game=1, c_puct_init=2.5, iters_hint=200)
        eng.attach_nets(nets)
        eng.set_tree_nets(m1)
        if eng.new_roots() > 0:
            eng.eval_net()
            eng.expand()
        eng.run_begin([120] * 8)
        eng.rounds_net(12)                       # round 1 eager, round 2 captures, rounds 3.. replay
        if switch:
            eng.set_tree_nets(m2)
        eng.rounds_net(60)
        vis, val, info = eng.root_dense()
        assert eng.status() == 0
        eng.close()
        for n in nets:
            n.close()
        return vis.copy(), val.copy(), info.copy()

    a, b, c = run(True, True), run(False, True), run(True, False)
    assert int(a[2][:, 2].min()) == 72
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    assert not np.array_equal(a[0], c[0])


def _usable_with_one_net(eng, net):
    net.attach(eng)
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([20] * eng.n_trees)
    while eng.remaining() > 0:
        eng.rounds_net(8)
    assert eng.status() == 0
    assert eng.root_dense()[2][:, 2].min() == 20


def test_errors_are_loud_and_leave_the_engine_usable():
    c4 = spec_of("connect4")
    a, b = Net(c4, netspec.init_weights(c4, seed=2), max_batch=8), Net(c4, netspec.init_weights(c4, seed=3), max_batch=8)
    gk = Net(spec_of("tictactoe"), netspec.init_weights(spec_of("tictactoe"), seed=2), max_batch=8)

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    with pytest.raises(EngineError, match="different games"):
        eng.attach_nets([a, gk])
    _usable_with_one_net(eng, a)
    eng.close()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    with pytest.raises(EngineError, match="tree_net"):
        eng.set_tree_nets([0, 1, 0, 0])              # one network attached
    eng.attach_nets([a, b])
    with pytest.raises(EngineError, match="tree_net"):
        eng.set_tree_nets([0, 1, 2, 0])
    _usable_with_one_net(eng, a)
    eng.close()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.enable_eval_cache(4096)
    with pytest.raises(EngineError, match="evaluation cache"):
        eng.attach_nets([a, b])
    _usable_with_one_net(eng, a)
    eng.close()
    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.attach_nets([a, b])
    with pytest.raises(EngineError, match="evaluation cache"):
        eng.enable_eval_cache(4096)
    _usable_with_one_net(eng, a)
    eng.close()

    build, train = _configs(use_gumbel=True)
    spec = net_spec_from_configs("connect4", build, train)
    W = netspec.init_weights(spec, seed=1)
    with pytest.raises(ValueError, match="Gumbel|gumbel"):
        BatchedSelfPlay(G.Connect4, build, train, range(2), 2, spec=spec, weights=W, opponent=(spec, W))
    for n in (a, b, gk):
        n.close()


def _configs(**kw):
    tc = dict(MCTS_iteration_limit=40, use_gumbel=False, c_puct_init=2.5, dirichlet_alpha=0.5, max_actions=42,
              num_explore_actions_first=2, num_explore_actions_second=2, games_per_gpu=64)
    tc.update(kw)
    return {"use_stablemax": False, "num_resnet_layers": 2}, tc


def _weights(seed, game="connect4"):
    build, train = _configs()
    return netspec.init_weights(net_spec_from_configs(game, build, train), seed=seed)


def test_match_of_identical_networks_is_an_exact_tie():
    W = _weights(1)
    r = arena.play_match(G.Connect4, _configs(), W, {k: v.copy() for k, v in W.items()}, 12, seed=3, n_slots=12)
    assert len(r["games"]) == 12
    for i in range(0, 12, 2):
        g0, g1 = r["games"][i], r["games"][i + 1]
        assert g0["opening"] == g1["opening"] and g0["a_first"] and not g1["a_first"]
        assert g0["actions"] == g1["actions"] and g0["winner"] == g1["winner"]
    assert r["score"] == 0.5
    assert r["wins"] == r["losses"]


def _replay_and_check(r, cls, max_actions):
    name = G.game_name_of(cls())
    for g in r["games"]:
        game = cls()
        plies = g["opening"] + g["actions"]
        assert g["length"] == len(plies)
        w = -2
        for j, a in enumerate(plies):
            assert w == -2, g
            game.do_action(G.id_to_action(name, a))
            w = int(game.check_win())
        if len(plies) >= max_actions:
            assert g["winner"] == 0, g                  # the max_actions cut-off is a draw
        else:
            assert w != -2 and g["winner"] == w, g


def test_match_of_different_networks():
    build, train = _configs()
    Wa, Wb = _weights(1), _weights(7)
    r8 = arena.play_match(G.Connect4, (build, train), Wa, Wb, 16, seed=5, n_slots=8)
    r64 = arena.play_match(G.Connect4, (build, train), Wa, Wb, 16, seed=5, n_slots=64)
    assert r8["games"] == r64["games"]                  # routing under different batch layouts gives the same games
    assert r8["wins"] + r8["draws"] + r8["losses"] == 16
    assert r8["score"] == (r8["wins"] + 0.5 * r8["draws"]) / 16
    _replay_and_check(r8, G.Connect4, train["max_actions"])
    assert len({tuple(g["opening"]) for g in r8["games"]}) > 1

    ia, ib = 5, 40                                      # 5 < 7 legal moves: the 3 * n_legal rule (MCTS.py:543-546)
    r = arena.play_match(G.Connect4, (build, train), Wa, Wb, 8, seed=9, iterations=(ia, ib), n_slots=8)
    _replay_and_check(r, G.Connect4, train["max_actions"])
    for g in r["games"]:
        game = G.Connect4()
        for a in g["opening"]:
            game.do_action(G.id_to_action("connect4", a))
        a_player = -1 if g["a_first"] else 1
        for a, its in zip(g["actions"], g["iterations"]):
            n_legal = len(game.get_legal_actions())
            lim = ia if game.get_next_player() == a_player else ib
            want = 1 if n_legal == 1 else (3 * n_legal if lim < n_legal else lim)
            assert its == want, (g, a, its, want)
            game.do_action(G.id_to_action("connect4", a))
