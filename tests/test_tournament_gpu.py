"""GPU suite: up to eight networks attached to one engine (K-way leaf routing), networks sharing an activation workspace
(gaz_net_create_shared) and the tournament driver (arena.play_tournament)."""
import ctypes as C

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


def spec_of(game, **kw):
    return netspec.build_spec(game, "softmax", **dict(SPECS[game], **kw))


def search(game, nets, tree_net, n_games, iters, seed=0, max_plies=6):
    """n_games random positions, one tree each, searched to `iters` with graph-replayed rounds; nets = [A] attaches A
    alone, otherwise all of them with tree t on nets[tree_net[t]].  Returns root_dense (visits, value sums, info)."""
    eng = Engine(game, n_games=n_games, mode="puct", trees_per_game=1, c_puct_init=2.5, iters_hint=iters)
    if len(nets) == 1:
        nets[0].attach(eng)
    else:
        eng.attach_nets(nets)
        eng.set_tree_nets(tree_net)
    rng = np.random.RandomState(seed)
    for i in range(n_games):
        g = ep.random_position(game, rng, rng.randint(0, max_plies))
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


def assert_same(got, ref):
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1].view(np.uint32), ref[1].view(np.uint32))
    np.testing.assert_array_equal(got[2], ref[2])


@pytest.mark.parametrize("K", [3, 5, 8])
@pytest.mark.parametrize("game", ["tictactoe", "connect4", "gomoku"])
def test_k_copies_are_invisible(game, K):
    """K networks with the same weights: routing every tree's leaves through any of them changes no bit of the search.
    max_batch 16 < 40 trees, so every network runs three chunks per round (a graph key wider than 32 bits at K = 8)."""
    spec = spec_of(game)
    W = netspec.init_weights(spec, seed=3)
    n_games, iters = 40, 60
    ref_net = Net(spec, W, max_batch=16)
    ref = search(game, [ref_net], None, n_games, iters)
    nets = []
    for k in range(K):     # K = 3: independent workspaces; 5 and 8: one shared workspace
        nets.append(Net(spec, W, max_batch=16, share=nets[0] if (K > 3 and k > 0) else None))
    rng = np.random.RandomState(K)
    no_one = rng.randint(0, K - 1, n_games)
    no_one[no_one >= 1] += 1                            # network 1 serves no tree
    for mapping in (rng.randint(0, K, n_games), np.full(n_games, K - 1), no_one):
        assert_same(search(game, nets, mapping, n_games, iters), ref)
    for n in nets + [ref_net]:
        n.close()


def test_k_copies_are_invisible_across_routing_tiles():
    """TicTacToe, 2085 trees (more than two 1024-leaf routing tiles, not a multiple of 32): the per-network carries cross
    tiles; 4 chunks of 600 per network and round."""
    spec = spec_of("tictactoe")
    W = netspec.init_weights(spec, seed=4)
    n_games, iters = 2085, 30
    ref_net = Net(spec, W, max_batch=600)
    ref = search("tictactoe", [ref_net], None, n_games, iters, max_plies=4)
    nets = [Net(spec, W, max_batch=600)]
    nets += [Net(spec, W, max_batch=600, share=nets[0]) for _ in range(5)]
    mapping = np.random.RandomState(9).randint(0, 6, n_games)
    assert_same(search("tictactoe", nets, mapping, n_games, iters, max_plies=4), ref)
    for n in nets + [ref_net]:
        n.close()


@pytest.mark.parametrize("game,iters", [("connect4", 120), ("gomoku", 150)])
def test_each_tree_searches_with_its_own_network(game, iters):
    """Four networks with different weights and a random mapping: every tree's root statistics equal the C oracle's
    search with the host forward of that tree's network as its evaluator."""
    spec = spec_of(game)
    nets = []
    for k, seed in enumerate((2, 5, 8, 11)):
        nets.append(Net(spec, netspec.init_weights(spec, seed=seed), max_batch=4, share=nets[0] if k else None))
    n_games = 14
    mapping = np.random.RandomState(4).randint(0, 4, n_games).astype(np.uint8)
    mapping[:4] = [0, 1, 2, 3]
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


def test_a_k4_remapping_survives_graph_replay():
    """set_tree_nets after the round graph was captured, four networks: the replayed graph (run A) equals eager rounds
    (run B, Net.profile on); run C keeps the first mapping and differs."""
    spec = spec_of("connect4")
    Ws = [netspec.init_weights(spec, seed=s) for s in (2, 6, 7, 9)]
    m1 = np.array([0, 1, 2, 3] * 3, np.uint8)
    m2 = np.array([3, 2, 0, 1, 1, 3, 2, 0, 2, 0, 3, 1], np.uint8)

    def run(graph, switch):
        nets = []
        for W in Ws:
            nets.append(Net(spec, W, max_batch=4, share=nets[0] if nets else None))
        if not graph:
            for n in nets:
                n.profile(16384)
        eng = Engine("connect4", n_games=12, mode="puct", trees_per_game=1, c_puct_init=2.5, iters_hint=200)
        eng.attach_nets(nets)
        eng.set_tree_nets(m1)
        if eng.new_roots() > 0:
            eng.eval_net()
            eng.expand()
        eng.run_begin([120] * 12)
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


@pytest.mark.parametrize("game", ["connect4", "gomoku"])
def test_shared_workspace_forward_is_bit_identical(game):
    spec = spec_of(game)
    Wa, Wb = netspec.init_weights(spec, seed=1), netspec.init_weights(spec, seed=2)
    a = Net(spec, Wa, max_batch=64)
    b = Net(spec, Wb, max_batch=64, share=a)
    b_own, a_own = Net(spec, Wb, max_batch=64), Net(spec, Wa, max_batch=64)
    rng = np.random.RandomState(0)
    xs = [np.stack([ep.random_position(game, rng, rng.randint(0, 10)).input_state() for _ in range(n)]) for n in (64, 37, 5)]
    for x in xs:            # A, B, A interleaved on one workspace
        pa, va = a.forward(x)
        pb, vb = b.forward(x)
        pa2, va2 = a.forward(x)
        qa, wa = a_own.forward(x)
        qb, wb = b_own.forward(x)
        for got, want in ((pa, qa), (va, wa), (pb, qb), (vb, wb), (pa2, qa), (va2, wa)):
            np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    # the sharer counts its weights and tables, not the activations
    ws = a.bytes_allocated() - b.bytes_allocated()
    assert b.bytes_allocated() == b_own.bytes_allocated() - ws
    rows = 64 * (64 if game == "connect4" else 256)     # padded rows of 64 boards
    assert ws >= rows * 64 * 2                          # at least one bf16 activation buffer of 64 channels
    # closing the creator of the workspace first leaves the sharer working
    a.close()
    pb, vb = b.forward(xs[1])
    qb, wb = b_own.forward(xs[1])
    np.testing.assert_array_equal(pb.view(np.uint32), qb.view(np.uint32))
    np.testing.assert_array_equal(vb.view(np.uint32), wb.view(np.uint32))
    for n in (b, b_own, a_own):
        n.close()


def test_shared_workspace_refuses_a_different_structure():
    spec = spec_of("connect4")
    a = Net(spec, netspec.init_weights(spec, seed=1), max_batch=16)
    other = spec_of("connect4", num_blocks=3)
    with pytest.raises(EngineError, match="shared workspace"):
        Net(other, netspec.init_weights(other, seed=1), max_batch=16, share=a)
    with pytest.raises(EngineError, match="max_batch"):
        Net(spec, netspec.init_weights(spec, seed=1), max_batch=32, share=a)
    ttt = spec_of("tictactoe")
    with pytest.raises(EngineError, match="game"):
        Net(ttt, netspec.init_weights(ttt, seed=1), max_batch=16, share=a)
    b = Net(spec, netspec.init_weights(spec, seed=2), max_batch=16, share=a)   # a still shares after the refusals
    x = np.zeros((3, 6, 7, 4), np.int8)
    assert np.isfinite(b.forward(x)[1]).all()
    a.close(); b.close()


def test_batched_self_play_with_eight_networks_allocates_one_workspace():
    build, train = _configs(game="gomoku")
    spec = net_spec_from_configs("gomoku", build, train)
    Ws = [netspec.init_weights(spec, seed=s) for s in range(8)]
    pairs = arena.round_robin(8)
    sp = BatchedSelfPlay(G.Gomoku, build, train, range(28 * 2), 64, spec=spec, weights=Ws[0], use_noise=False,
                         opponents=[(spec, W) for W in Ws[1:]], tree_nets=arena.tournament_tree_nets(pairs, 2))
    try:
        own = [n.bytes_allocated() for n in sp.nets]
        assert len(sp.nets) == 8 and len(set(own[1:])) == 1
        ws = own[0] - own[1]
        independent = Net(spec, Ws[0], max_batch=sp.n_slots)
        assert independent.bytes_allocated() == own[0]
        independent.close()
        assert sum(own) == ws + 8 * own[1]               # one workspace + 8 weight sets
        assert ws > 0
    finally:
        sp.close()


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
    nets = [Net(c4, netspec.init_weights(c4, seed=s), max_batch=8) for s in range(9)]
    ttt = Net(spec_of("tictactoe"), netspec.init_weights(spec_of("tictactoe"), seed=2), max_batch=8)

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    with pytest.raises(EngineError, match="1 to 8"):
        eng.attach_nets(nets)                                   # 9 networks
    with pytest.raises(EngineError, match="different games"):
        eng.attach_nets(nets[:2] + [ttt])
    hs = (C.c_void_p * 3)(nets[0]._h.value, None, nets[1]._h.value)
    assert eng.lib.gaz_attach_nets(eng._h, hs, 3) < 0
    assert "null" in eng.lib.gaz_last_error().decode()
    _usable_with_one_net(eng, nets[0])
    eng.close()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.attach_nets(nets[:3])
    with pytest.raises(EngineError, match="tree_net"):
        eng.set_tree_nets([0, 1, 3, 0])
    _usable_with_one_net(eng, nets[0])
    eng.close()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.enable_eval_cache(4096)
    with pytest.raises(EngineError, match="evaluation cache"):
        eng.attach_nets(nets[:5])
    _usable_with_one_net(eng, nets[0])
    eng.close()
    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.attach_nets(nets[:8])
    with pytest.raises(EngineError, match="evaluation cache"):
        eng.enable_eval_cache(4096)
    _usable_with_one_net(eng, nets[0])
    eng.close()

    # a table naming network 7 and then only two networks attached: the table is back on network 0, and the search runs
    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.attach_nets(nets[:8])
    eng.set_tree_nets([7, 6, 1, 0])
    eng.attach_nets(nets[:2])
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([20] * 4)
    while eng.remaining() > 0:
        eng.rounds_net(8)
    assert eng.status() == 0 and eng.root_dense()[2][:, 2].min() == 20
    eng.close()
    for n in nets + [ttt]:
        n.close()


def _configs(game="connect4", **kw):
    tc = dict(MCTS_iteration_limit=40, use_gumbel=False, c_puct_init=2.5, dirichlet_alpha=0.5,
              max_actions=42 if game == "connect4" else 60, num_explore_actions_first=2, num_explore_actions_second=2,
              games_per_gpu=64)
    tc.update(kw)
    return {"use_stablemax": False, "num_resnet_layers": 2}, tc


def _weights(seed, game="connect4"):
    build, train = _configs(game)
    return netspec.init_weights(net_spec_from_configs(game, build, train), seed=seed)


def test_a_tournament_is_the_union_of_its_matches():
    build, train = _configs()
    Ws = [_weights(1), _weights(7), _weights(4)]
    r = arena.play_tournament(G.Connect4, (build, train), Ws, 8, seed=5, n_slots=10)   # 10 < 24: pairs reseat mixed
    assert [(p["i"], p["j"]) for p in r["pairs"]] == [(0, 1), (0, 2), (1, 2)]
    assert len(r["games"]) == 24
    for p, (i, j) in enumerate(arena.round_robin(3)):
        m = arena.play_match(G.Connect4, (build, train), Ws[i], Ws[j], 8, seed=5, n_slots=8)
        mine = [g for g in r["games"] if g["pair"] == p]
        assert [g["game_id"] - 8 * p for g in mine] == [g["game_id"] for g in m["games"]]
        for t, g in zip(mine, m["games"]):
            assert t["first"] == (i if g["a_first"] else j) and t["second"] == (j if g["a_first"] else i)
            for k in ("opening", "actions", "winner", "length", "iterations"):
                assert t[k] == g[k], (p, k, t, g)
        pr = r["pairs"][p]
        for k in ("wins", "draws", "losses", "score", "elo", "elo_ci"):
            assert pr[k] == m[k], k
        assert pr["by_colour"]["i_first"] == m["by_colour"]["a_first"]
        assert pr["by_colour"]["i_second"] == m["by_colour"]["a_second"]
        assert r["crosstable"][i][j] == m["score"] and r["crosstable"][j][i] == 1.0 - m["score"]
    assert all(np.isnan(r["crosstable"][k][k]) for k in range(3))
    if r["ratings"] is None:
        assert r["ratings_reason"]
    else:
        assert r["ratings"]["elo"][0] == 0.0 and len(r["ratings"]["elo_ci"]) == 3


def test_gauntlet_and_per_network_iteration_limits():
    build, train = _configs()
    Ws = [_weights(1), _weights(7), _weights(4)]
    lims = (5, 40, 12)                                  # 5 < 7 legal moves: the 3 * n_legal rule (MCTS.py:543-546)
    r = arena.play_tournament(G.Connect4, (build, train), Ws, 4, pairs=arena.gauntlet(3), iterations=lims, seed=9,
                              n_slots=8)
    assert [(p["i"], p["j"]) for p in r["pairs"]] == [(0, 1), (0, 2)]
    assert np.isnan(r["crosstable"][1][2]) and np.isnan(r["crosstable"][2][1])
    assert len(r["games"]) == 8
    for g in r["games"]:
        game = G.Connect4()
        for a in g["opening"]:
            game.do_action(G.id_to_action("connect4", a))
        for a, its in zip(g["actions"], g["iterations"]):
            n_legal = len(game.get_legal_actions())
            who = g["first"] if game.get_next_player() == -1 else g["second"]
            lim = lims[who]
            want = 1 if n_legal == 1 else (3 * n_legal if lim < n_legal else lim)
            assert its == want, (g, a, its, want)
            game.do_action(G.id_to_action("connect4", a))
        if g["length"] >= train["max_actions"]:
            assert g["winner"] == 0                  # the max_actions cut-off is a draw
        else:
            assert g["winner"] == int(game.check_win()) != -2


def test_identical_networks_tie():
    W = _weights(1)
    r = arena.play_tournament(G.Connect4, _configs(), [W, {k: v.copy() for k, v in W.items()}, W], 6, seed=3, n_slots=12)
    for p in r["pairs"]:
        assert p["score"] == 0.5 and p["wins"] == p["losses"]
    assert r["ratings"] is not None, r["ratings_reason"]
    assert r["ratings"]["elo"] == [0.0, 0.0, 0.0]
