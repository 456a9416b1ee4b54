"""GPU suite: symmetric network evaluation (gaz_set_eval_symmetry / Engine.set_eval_symmetry).  The C oracle's evaluator
restates both modes on the host: RANDOM forwards the state gathered through the symmetry that the Python twin of the device
hash draws and maps the row back; ENSEMBLE averages the n mapped-back rows in g order.  Forward rows do not depend on their
batch position, so every comparison is bit-exact."""
import ctypes as C

import numpy as np
import pytest

import engine_parity as ep
import oracle as orc
import sym_hash
from grok_alpha_zero_b200 import arena, netspec
from grok_alpha_zero_b200 import games as G
from grok_alpha_zero_b200.Self_Play import BatchedSelfPlay, net_spec_from_configs
from grok_alpha_zero_b200.engine import DIMS, Engine, EngineError
from grok_alpha_zero_b200.net import Net

pytestmark = pytest.mark.gpu

SPECS = {"tictactoe": {}, "connect4": dict(num_blocks=2), "gomoku": dict(num_blocks=2, use_se=True)}
GAMES = ["tictactoe", "connect4", "gomoku"]
SEED = 0x5EED5EED1234


def spec_of(game, head="softmax"):
    return netspec.build_spec(game, head, **SPECS[game])


def positions(game, n, seed=0, max_plies=8):
    rng = np.random.RandomState(seed)
    return [ep.random_position(game, rng, rng.randint(0, max_plies)) for _ in range(n)]


def host_evaluator(net, game, mode, key=None, seed=SEED):
    """the device's symmetric evaluation of one request, restated with host forwards"""
    H, W, Cc, P = DIMS[game]
    ps, pp = G.eval_symmetries(game)
    n = len(ps)

    def ev(state):
        s = np.asarray(state, np.int8).reshape(-1)
        if mode == "random":
            g = sym_hash.sym_draw(s, seed, key, n)
            p, v = net.forward(s[ps[g]].reshape(1, H, W, Cc))
            return p[0][pp[g]], v[0]
        pol, val = np.zeros(P, np.float32), np.float32(0.0)
        for g in range(n):                    # one row per forward: the network's max_batch may be below n
            p, v = net.forward(s[ps[g]].reshape(1, H, W, Cc))
            pol = (pol + p[0][pp[g]]).astype(np.float32)
            val = np.float32(val + v[0])
        inv = np.float32(1.0) / np.float32(n)
        return (pol * inv).astype(np.float32), np.float32(val * inv)
    return ev


def run_engine(game, nets, games, iters, mode=None, tree_net=None, keys=None, midway=None, gumbel=False, profile=False,
               **kw):
    """one tree per position; mode None never calls the setter.  midway(eng) runs after the first 16 rounds (by then the
    round graph is captured and replayed).  Returns root_dense."""
    n = len(games)
    eng = Engine(game, n_games=n, mode="gumbel" if gumbel else "puct", trees_per_game=1, c_puct_init=2.5,
                 iters_hint=iters * (4 if gumbel else 1), **kw)
    if profile:
        for net in nets:
            net.profile(16384)
    if len(nets) == 1:
        nets[0].attach(eng)
    else:
        eng.attach_nets(nets)
        eng.set_tree_nets(tree_net)
    if keys is not None:
        eng.set_tree_keys(keys)
    if mode is not None:
        eng.set_eval_symmetry(mode, SEED)
    for i, g in enumerate(games):
        eng.set_game(i, g.board, g.next_player, g.history)
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([iters] * n)
    eng.rounds_net(16)
    if midway is not None:
        midway(eng)
    while eng.remaining() > 0:
        eng.rounds_net(16)
    assert eng.status() == 0
    out = eng.root_dense()
    if profile:
        for net in nets:
            net.profile(0)
    eng.close()
    return out


def assert_same(got, ref):
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1].view(np.uint32), ref[1].view(np.uint32))
    np.testing.assert_array_equal(got[2], ref[2])


def check_vs_oracle(game, net, games, iters, mode, keys=None, gumbel=False, activation_fn="softmax", **kw):
    n = len(games)
    eng = Engine(game, n_games=n, mode="gumbel" if gumbel else "puct", trees_per_game=1, c_puct_init=2.5,
                 iters_hint=iters * (4 if gumbel else 1), activation_fn=activation_fn, **kw)
    net.attach(eng)
    if keys is not None:
        eng.set_tree_keys(keys)
    eng.set_eval_symmetry(mode, SEED)
    for i, g in enumerate(games):
        eng.set_game(i, g.board, g.next_player, g.history)
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([iters] * n)
    while eng.remaining() > 0:
        eng.rounds_net(16)
    assert eng.status() == 0
    for i, g in enumerate(games):
        key = sym_hash.tree_key(SEED, i, keys)
        t = orc.OracleTree(game, gumbel, evaluator=host_evaluator(net, game, mode, key), c_puct_init=2.5,
                           activation_fn=activation_fn)
        t.new_root(g)
        t.run(iters)
        ref, st = t.root_stats(), eng.root_stats(i)
        where = "%s %s tree %d" % (game, mode, i)
        np.testing.assert_array_equal(st["action"], ref["action"], err_msg=where)
        np.testing.assert_array_equal(st["visits"], ref["visits"], err_msg=where)
        np.testing.assert_array_equal(st["values"].view(np.uint32), ref["values"].view(np.uint32), err_msg=where)
        assert st["evals"] == t.n_evals, where
    eng.close()


@pytest.mark.parametrize("game", GAMES)
def test_off_means_off(game):
    """RANDOM set and then NONE again, before the search or after the round graph was captured: bit-identical to an engine
    that never called the setter"""
    spec = spec_of(game)
    net = Net(spec, netspec.init_weights(spec, seed=1), max_batch=32)
    games = positions(game, 20)
    ref = run_engine(game, [net], games, 80)

    def flip(eng):
        eng.set_eval_symmetry("random", 7)
        eng.set_eval_symmetry("none")

    assert_same(run_engine(game, [net], games, 80, midway=flip), ref)
    eng_first = run_engine(game, [net], games, 80, mode="random", midway=lambda e: None)
    assert not np.array_equal(eng_first[0], ref[0])           # the mode does change the search
    assert_same(run_engine(game, [net], games, 80, mode="none"), ref)
    net.close()


@pytest.mark.parametrize("game", GAMES)
def test_random_matches_the_oracle(game):
    spec = spec_of(game)
    net = Net(spec, netspec.init_weights(spec, seed=2), max_batch=8)
    games = positions(game, 12, seed=3)
    check_vs_oracle(game, net, games, 100, "random")
    keys = np.random.RandomState(5).randint(0, 2**62, len(games)).astype(np.uint64) * np.uint64(3)
    check_vs_oracle(game, net, games, 100, "random", keys=keys)
    net.close()


@pytest.mark.parametrize("game", GAMES)
def test_ensemble_matches_the_oracle(game):
    spec = spec_of(game)
    net = Net(spec, netspec.init_weights(spec, seed=4), max_batch=128)
    check_vs_oracle(game, net, positions(game, 12, seed=6), 100, "ensemble")
    net.close()


def test_ensemble_gumbel_stablemax_averages_logits():
    """Gumbel search with StableMax over the linear head: ENSEMBLE averages the logit rows"""
    spec = spec_of("gomoku", "linear")
    net = Net(spec, netspec.init_weights(spec, seed=8), max_batch=64)
    check_vs_oracle("gomoku", net, positions("gomoku", 6, seed=2, max_plies=12), 64, "ensemble", gumbel=True,
                    activation_fn="stablemax")
    check_vs_oracle("gomoku", net, positions("gomoku", 6, seed=4, max_plies=12), 64, "random", gumbel=True,
                    activation_fn="stablemax")
    net.close()


@pytest.mark.parametrize("game", ["connect4", "gomoku"])
def test_ensemble_in_many_chunks_matches_the_oracle(game):
    """max_batch 5 < n_sym x 12 leaves: 20 (Gomoku) or 5 (Connect4) chunks per evaluation"""
    spec = spec_of(game)
    net = Net(spec, netspec.init_weights(spec, seed=9), max_batch=5)
    check_vs_oracle(game, net, positions(game, 12, seed=8), 60, "ensemble")
    net.close()


def test_round_graph_replay_equals_eager_rounds_and_a_mode_change_after_capture_takes_effect():
    spec = spec_of("connect4")
    W = netspec.init_weights(spec, seed=3)
    games = positions("connect4", 12, seed=1)

    def run(graph, switch):
        net = Net(spec, W, max_batch=8)
        out = run_engine("connect4", [net], games, 120, mode="random", profile=not graph,
                         midway=(lambda e: e.set_eval_symmetry("ensemble", SEED)) if switch else None)
        net.close()
        return out

    a, b, c = run(True, True), run(False, True), run(True, False)
    assert_same(a, b)
    assert not np.array_equal(a[0], c[0])


@pytest.mark.parametrize("mode", ["random", "ensemble"])
@pytest.mark.parametrize("game", GAMES)
def test_k_copies_with_symmetry_are_invisible(game, mode):
    spec = spec_of(game)
    W = netspec.init_weights(spec, seed=5)
    games = positions(game, 24, seed=2)
    ref_net = Net(spec, W, max_batch=16)
    ref = run_engine(game, [ref_net], games, 60, mode=mode)
    nets = [Net(spec, W, max_batch=16)]
    nets += [Net(spec, W, max_batch=16, share=nets[0]) for _ in range(2)]
    rng = np.random.RandomState(1)
    for mapping in (rng.randint(0, 3, len(games)), np.full(len(games), 2)):
        assert_same(run_engine(game, nets, games, 60, mode=mode, tree_net=mapping.astype(np.uint8)), ref)
    for n in nets + [ref_net]:
        n.close()


def _configs(**kw):
    tc = dict(MCTS_iteration_limit=30, use_gumbel=False, c_puct_init=2.5, dirichlet_alpha=0.5, max_actions=42,
              num_explore_actions_first=2, num_explore_actions_second=2, games_per_gpu=64)
    tc.update(kw)
    return {"use_stablemax": False, "num_resnet_layers": 2}, tc


def test_self_play_with_random_symmetry_does_not_depend_on_the_layout():
    build, train = _configs(eval_symmetry="random")
    spec = net_spec_from_configs("connect4", build, train)
    W = netspec.init_weights(spec, seed=6)
    out = []
    for slots in (8, 64):
        sp = BatchedSelfPlay(G.Connect4, build, train, range(16), slots, spec=spec, weights=W, seed=13)
        try:
            out.append(sorted(sp.play(), key=lambda g: g["game_id"]))
        finally:
            sp.close()
    a, b = out
    assert [g["game_id"] for g in a] == list(range(16))
    for x, y in zip(a, b):
        assert x["winner"] == y["winner"] and x["length"] == y["length"]
        np.testing.assert_array_equal(x["states"], y["states"])
        np.testing.assert_array_equal(x["policies"].view(np.uint32), y["policies"].view(np.uint32))


def test_identical_networks_tie_with_the_ensemble():
    build, train = _configs()
    W = netspec.init_weights(net_spec_from_configs("connect4", build, train), seed=1)
    r = arena.play_match(G.Connect4, (build, train), W, {k: v.copy() for k, v in W.items()}, 8, seed=3, n_slots=8,
                         symmetry="ensemble")
    assert r["score"] == 0.5 and r["wins"] == r["losses"]


def _usable(eng, net):
    net.attach(eng)
    eng.set_eval_symmetry("none")
    if eng.new_roots() > 0:
        eng.eval_net()
        eng.expand()
    eng.run_begin([20] * eng.n_trees)
    while eng.remaining() > 0:
        eng.rounds_net(8)
    assert eng.status() == 0 and eng.root_dense()[2][:, 2].min() == 20


def test_refusals_are_loud_and_leave_the_engine_usable():
    spec = spec_of("connect4")
    net = Net(spec, netspec.init_weights(spec, seed=2), max_batch=8)
    ps, pp = G.eval_symmetries("connect4")

    def raw(eng, mode, n, a, b):
        rc = eng.lib.gaz_set_eval_symmetry(eng._h, mode, n, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), 0)
        return rc, eng.lib.gaz_last_error().decode()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.enable_eval_cache(4096)
    with pytest.raises(EngineError, match="evaluation cache"):
        eng.set_eval_symmetry("random")
    _usable(eng, net)
    eng.close()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    eng.set_eval_symmetry("ensemble")
    with pytest.raises(EngineError, match="evaluation cache"):
        eng.enable_eval_cache(4096)
    _usable(eng, net)                       # back to NONE: now the cache may be enabled
    eng.enable_eval_cache(4096)
    eng.close()

    eng = Engine("connect4", n_games=4, mode="puct", trees_per_game=1, iters_hint=100)
    bad = ps.copy()
    bad[1][3] = bad[1][4]
    rc, msg = raw(eng, 1, 2, bad, pp)
    assert rc < 0 and "permutation" in msg
    badp = pp.copy()
    badp[1][0] = 7
    rc, msg = raw(eng, 2, 2, ps, badp)
    assert rc < 0 and "permutation" in msg
    for n in (0, 9):
        rc, msg = raw(eng, 1, n, np.resize(ps, (max(n, 1), ps.shape[1])), np.resize(pp, (max(n, 1), pp.shape[1])))
        assert rc < 0 and "n_sym" in msg
    rc, msg = raw(eng, 3, 2, ps, pp)
    assert rc < 0 and "unknown symmetry mode" in msg
    with pytest.raises(EngineError, match="unknown eval symmetry"):
        eng.set_eval_symmetry("mirror")
    _usable(eng, net)
    eng.close()
    net.close()
