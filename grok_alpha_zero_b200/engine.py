"""Engine: thin host-side handle over the C ABI (include/gaz_b200.h).

All search state (trees, boards, priors, visit counts) lives in HBM; this class only moves
small control arrays.  `lib` is injectable so the CPU test-suite can drive the warp code
through the test-only host emulation; the package itself always passes the CUDA library.
"""
import ctypes as C

import numpy as np

from . import _lib

GAMES = {"tictactoe": 0, "connect4": 1, "gomoku": 2}
DIMS = {"tictactoe": (3, 3, 2, 9), "connect4": (6, 7, 4, 7), "gomoku": (15, 15, 2, 225)}  # H, W, C, P
TERM_NONE, TERM_DRAW, TERM_WIN = 0, 1, 2
SYM_MODES = {"none": 0, "random": 1, "ensemble": 2}   # GAZ_SYM_* of include/gaz_net.h


class EngineError(RuntimeError):
    pass


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_caps(game, iters, mode="puct"):
    """(node_cap, slot_cap) big enough for `iters` simulations per move with sub-tree reuse."""
    H, W, _, P = DIMS[game]
    L = P if game != "connect4" else 7
    nodes = int(iters * (2.2 if game == "gomoku" else 6.0)) + 4 * L + 64
    if mode == "gumbel":
        nodes = int(iters * 1.5) + 4 * L + 64
    slots = nodes * min(L, 225) + 256
    return nodes, slots


class Engine:
    def __init__(self, game, n_games=1, mode="puct", trees_per_game=1, node_cap=None, slot_cap=None,
                 c_puct_init=2.5, c_puct_base=19652.0, m=16, c_visit=50.0, c_scale=0.1, activation_fn="softmax",
                 device=0, lut_n=1 << 20, iters_hint=1200, lib=None, slot_pool=0):
        self.lib = lib if lib is not None else _lib.load()
        self.game = game
        self.H, self.W, self.C, self.P = DIMS[game]
        self.mode = mode
        self.n_games = n_games
        self.trees_per_game = trees_per_game
        self.n_trees = n_games * trees_per_game
        if node_cap is None or slot_cap is None:
            nc, sc = default_caps(game, iters_hint, mode)
            node_cap = node_cap or nc
            slot_cap = slot_cap or sc
        cfg = _lib.GazConfig(GAMES[game], 1 if mode == "gumbel" else 0, n_games, trees_per_game, node_cap, slot_cap,
                             device, lut_n, c_puct_init, c_puct_base, m, int(activation_fn == "softmax"),
                             c_visit, c_scale, int(slot_pool))
        self.node_cap, self.slot_cap = int(node_cap), int(slot_cap)
        h = C.c_void_p()
        self._h = None
        self._ck(self.lib.gaz_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.state_size = self.H * self.W * self.C

    # ------------------------------------------------------------------ utils
    def _ck(self, rc):
        if rc < 0:
            raise EngineError(self.lib.gaz_last_error().decode())
        return rc

    def close(self):
        if self._h is not None:
            self.lib.gaz_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------- game state
    def set_game(self, g, board, next_player, history):
        b = np.ascontiguousarray(np.asarray(board).reshape(-1), dtype=np.int8)
        tail = np.array(list(reversed(history[-3:])) + [0, 0, 0], dtype=np.int16)
        self._ck(self.lib.gaz_set_game(self._h, g, _p(b), int(next_player), _p(tail), len(history)))

    def set_games(self, boards, next_players, hist_lens=None, last3=None, last_actions=None):
        """Upload every live game at once: boards int8 (n_games, H, W) (pinned memory welcome)."""
        b = np.ascontiguousarray(boards, dtype=np.int8).reshape(self.n_games, self.H * self.W)
        meta = np.zeros((self.n_games, 4), dtype=np.int32)
        meta[:, 0] = next_players
        meta[:, 1] = (b != 0).sum(1) if hist_lens is None else hist_lens
        meta[:, 2] = 0 if last3 is None else last3
        meta[:, 3] = -1 if last_actions is None else last_actions
        self._keep = (b, meta)  # the copy is asynchronous
        self._ck(self.lib.gaz_set_games(self._h, _p(b), _p(meta)))

    def reset_games(self):
        self._ck(self.lib.gaz_reset_games(self._h))

    def apply_actions(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.int16)
        w = np.zeros(self.n_games, dtype=np.int32)
        self._ck(self.lib.gaz_apply_actions(self._h, _p(a), _p(w)))
        return w

    def get_states(self):
        """get_input_state() of every live game: (states int8 (n_games, H, W, C), info int32 (n_games, 4) =
        next_player, len(action_history), winner (-2 running), last action id)"""
        st = np.zeros((self.n_games, self.H, self.W, self.C), dtype=np.int8)
        info = np.zeros((self.n_games, 4), dtype=np.int32)
        self._ck(self.lib.gaz_get_states(self._h, _p(st), _p(info)))
        return st, info

    def set_noise(self, dirichlet_alpha, dirichlet_epsilon, seed=0):
        self._ck(self.lib.gaz_set_noise(self._h, float(dirichlet_alpha), float(dirichlet_epsilon), int(seed)))

    def set_tree_keys(self, keys):
        k = None if keys is None else np.ascontiguousarray(keys, dtype=np.uint64)
        self._ck(self.lib.gaz_set_tree_keys(self._h, _p(k)))

    def gumbel_pi_dense(self):
        pi = np.zeros((self.n_trees, self.P), dtype=np.float32)
        self._ck(self.lib.gaz_gumbel_pi_dense(self._h, _p(pi)))
        return pi

    def get_game(self, g):
        b = np.zeros(self.H * self.W, dtype=np.int8)
        info = np.zeros(3, dtype=np.int32)
        self._ck(self.lib.gaz_get_game(self._h, g, _p(b), _p(info)))
        return b.reshape(self.H, self.W), int(info[0]), int(info[1]), int(info[2])

    # ----------------------------------------------------------------- search
    def set_puct_params(self, c_puct_init, c_puct_base):
        self._ck(self.lib.gaz_set_puct_params(self._h, c_puct_init, c_puct_base))

    def set_gumbel_params(self, m, c_visit, c_scale, use_softmax):
        self._ck(self.lib.gaz_set_gumbel_params(self._h, int(m), float(c_visit), float(c_scale), int(use_softmax)))

    def new_roots(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        return self._ck(self.lib.gaz_new_roots(self._h, _p(m)))

    def run_begin(self, limits):
        lim = np.ascontiguousarray(np.broadcast_to(np.asarray(limits, dtype=np.int32), (self.n_trees,)))
        self._ck(self.lib.gaz_run_begin(self._h, _p(lim)))

    def select(self):
        return self._ck(self.lib.gaz_select(self._h))

    def get_leaves(self, n=None):
        cap = self.n_trees if n is None else n
        st = np.zeros((cap, self.H, self.W, self.C), dtype=np.int8)
        tr = np.zeros(cap, dtype=np.int32)
        k = self._ck(self.lib.gaz_get_leaves(self._h, _p(st), _p(tr)))
        return st[:k], tr[:k]

    def get_leaf_depths(self, n=None):
        """`depth` of every outstanding request as MCTS._compute_outputs passes it to a caching session"""
        d = np.zeros(self.n_trees if n is None else n, dtype=np.int32)
        k = self._ck(self.lib.gaz_get_leaf_depths(self._h, _p(d)))
        return d[:k]

    def put_evals(self, policy, value):
        p = np.ascontiguousarray(policy, dtype=np.float32).reshape(-1, self.P)
        v = np.ascontiguousarray(value, dtype=np.float32).reshape(-1)
        self._ck(self.lib.gaz_put_evals(self._h, _p(p), _p(v), p.shape[0]))

    def eval_hash(self, salt=0, logits=False):
        self._ck(self.lib.gaz_eval_hash(self._h, salt, int(logits)))

    def expand(self):
        self._ck(self.lib.gaz_expand(self._h))

    def remaining(self):
        return self._ck(self.lib.gaz_remaining(self._h))

    def rounds_hash(self, n, salt=0, logits=False):
        self._ck(self.lib.gaz_rounds_hash(self._h, n, salt, int(logits)))

    def prune(self, actions, create_new_root=False):
        a = np.ascontiguousarray(np.broadcast_to(np.asarray(actions, dtype=np.int16), (self.n_trees,)))
        return self._ck(self.lib.gaz_prune(self._h, _p(a), int(create_new_root)))

    def set_gumbel_noise(self, noise):
        if noise is None:
            self._ck(self.lib.gaz_set_gumbel_noise(self._h, None))
            return
        buf = np.zeros((self.n_trees, 256), dtype=np.float64)
        noise = np.asarray(noise, dtype=np.float64).reshape(self.n_trees, -1)
        buf[:, :noise.shape[1]] = noise
        self._ck(self.lib.gaz_set_gumbel_noise(self._h, _p(buf)))

    def root_stats(self, tree=0):
        act = np.zeros(256, np.int16); vis = np.zeros(256, np.uint32); val = np.zeros(256, np.float32)
        pri = np.zeros(256, np.float32); raw = np.zeros(256, np.float32)
        term = np.zeros(256, np.int8); exp = np.zeros(256, np.int8); info = np.zeros(8, np.int64)
        L = self._ck(self.lib.gaz_root_stats(self._h, tree, _p(act), _p(vis), _p(val), _p(pri), _p(raw), _p(term),
                                             _p(exp), _p(info)))
        return dict(action=act[:L], visits=vis[:L], values=val[:L], prior=pri[:L], raw=raw[:L], term=term[:L],
                    expanded=exp[:L], L=L, n_expanded=int(info[1]), root_visits=int(info[2]),
                    best_slot=int(info[3]), n_nodes=int(info[4]), n_slots=int(info[5]), iter=int(info[6]),
                    evals=int(info[7]))

    def root_dense(self, want_values=True):
        """Visit counts / value sums of every tree scattered by action id + per-tree info
        (root_visits, tau=0 move, iterations, evals)."""
        vis = np.zeros((self.n_trees, self.P), np.uint32)
        val = np.zeros((self.n_trees, self.P), np.float32) if want_values else None
        info = np.zeros((self.n_trees, 4), np.int32)
        self._ck(self.lib.gaz_root_dense(self._h, _p(vis), _p(val), _p(info)))
        return vis, val, info

    def timer_begin(self):
        self._ck(self.lib.gaz_timer_begin(self._h))

    def timer_end(self):
        ms = C.c_float()
        self._ck(self.lib.gaz_timer_end(self._h, C.byref(ms)))
        return float(ms.value)

    def sync(self):
        self._ck(self.lib.gaz_sync(self._h))

    def gumbel_pi(self, tree=0):
        pi = np.zeros(256, dtype=np.float32)
        self._ck(self.lib.gaz_gumbel_pi(self._h, tree, _p(pi)))
        return pi

    def eval_net(self):
        self._ck(self.lib.gaz_eval_net(self._h))

    def attach_nets(self, nets):
        """Attach 1 to 8 `net.Net` evaluators of this game.  With several, the leaves of tree t are served by
        nets[tree_net[t]] (set_tree_nets; every tree starts on network 0); the evaluation cache cannot be on."""
        nets = list(nets)
        hs = (C.c_void_p * len(nets))(*[n._h.value for n in nets])
        self._ck(self.lib.gaz_attach_nets(self._h, hs, len(nets)))
        self._net = nets  # keep alive

    def set_tree_nets(self, tree_net):
        """network index (< number of attached networks) of every tree, uint8 (n_trees,)"""
        t = np.ascontiguousarray(np.broadcast_to(np.asarray(tree_net), (self.n_trees,)), dtype=np.uint8)
        self._ck(self.lib.gaz_set_tree_nets(self._h, _p(t)))

    def set_eval_symmetry(self, mode, seed=0):
        """How the attached networks evaluate a request: "none" (default: once, as reached - the reference's behaviour),
        "random" (under one board symmetry drawn from a hash of seed, tree key and position) or "ensemble" (the mean of
        the outputs under all symmetries, mapped back; n times the network work).  Only "none" keeps reference parity.
        Tables: games.eval_symmetries.  Cannot be combined with the evaluation cache."""
        if mode not in SYM_MODES:
            raise EngineError("unknown eval symmetry %r (one of %s)" % (mode, ", ".join(SYM_MODES)))
        if SYM_MODES[mode] == 0:
            self._ck(self.lib.gaz_set_eval_symmetry(self._h, 0, 0, None, None, 0))
            return
        from .games import eval_symmetries
        ps, pp = eval_symmetries(self.game)
        self._ck(self.lib.gaz_set_eval_symmetry(self._h, SYM_MODES[mode], ps.shape[0], _p(ps), _p(pp), int(seed) & (2**64 - 1)))

    def rounds_net(self, n, sync=True):
        fn = self.lib.gaz_rounds_net if sync else self.lib.gaz_rounds_net_async
        self._ck(fn(self._h, int(n)))

    def status(self):
        return self._ck(self.lib.gaz_status(self._h))

    def tree_sizes(self):
        """(n_trees, 2) int32: nodes and child slots in use per tree (pools of node_cap / slot_cap)"""
        out = np.zeros((self.n_trees, 2), dtype=np.int32)
        self._ck(self.lib.gaz_tree_sizes(self._h, _p(out)))
        return out

    def enable_eval_cache(self, entries, shared=False):
        """device-side evaluation cache (Session_Cache.Cache_Wrapper's role): identical positions are evaluated once"""
        self._ck(self.lib.gaz_eval_cache_enable(self._h, int(entries), int(bool(shared))))

    def eval_cache_stats(self):
        out = np.zeros(3, dtype=np.int64)
        self._ck(self.lib.gaz_eval_cache_stats(self._h, _p(out)))
        return dict(lookups=int(out[0]), hits=int(out[1]), entries=int(out[2]))

    def pool_info(self):
        """slot page pool: dict(pages, free, page_slots, max_pages_per_tree)"""
        out = np.zeros(4, dtype=np.int64)
        self._ck(self.lib.gaz_pool_info(self._h, _p(out)))
        return dict(pages=int(out[0]), free=int(out[1]), page_slots=int(out[2]), max_pages_per_tree=int(out[3]))

    def bytes_allocated(self):
        return int(self.lib.gaz_bytes_allocated(self._h))

    # ------------------------------------------------- host-evaluator driving
    def eval_pending(self, evaluator):
        """Serve the outstanding leaf requests with a host evaluator
        (states int8 (n,H,W,C)) -> (policy (n,P) f32, value (n,) f32), then expand."""
        st, _ = self.get_leaves()
        if len(st):
            p, v = evaluator(st)
            self.put_evals(p, v)
        self.expand()
        return len(st)

    def run_host(self, limits, evaluator, max_rounds=1 << 30):
        """MCTS.run / MCTS_Gumbel.run for all trees, evaluator on the host."""
        self.run_begin(limits)
        rounds = 0
        while self.remaining() > 0 and rounds < max_rounds:
            n = self.select()
            if n > 0:
                self.eval_pending(evaluator)
            rounds += 1
        return rounds
