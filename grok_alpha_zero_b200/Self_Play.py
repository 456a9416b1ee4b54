"""Batched self-play on the B200 engine: the drop-in for `Self_Play.run_self_play` (Self_Play.py:259-413).

The reference runs one OS process per game (Self_Play.py:346-363), each looping `Self_Play.play` (:71-208).  Here
every GPU keeps thousands of games resident and advances them together, one move per outer iteration:

    get_input_state of every game  ->  MCTS.run / MCTS_Gumbel.run for every game (rounds of select -> network ->
    expand on the device)  ->  root statistics  ->  tau / opening-book move choice  ->  do_action + check_win  ->
    prune_tree on both trees (or a fresh Gumbel tree)  ->  finished games leave, queued games take their slots.

What is kept from `Self_Play.play`: two PUCT trees per game with the side to move searching `int(limit * 1.5)`
iterations (:97-106) or one Gumbel tree rebuilt every move (:110-112,151-153); tau = 1 for the first
`num_explore_actions_first/second` own moves, else 0 (:87-95); the opening book on move 0 (:130-140); the policy
target = scattered `[action, prob]` rows (:114), q target = win-rate of the played move (:117-125), z target and its
sign / draw rules (:127,159-170), value = 0.5 * (z + q) (:172), `max_actions` cut-off as a draw (:155-157), the
game's own `augment_sample` (:174), the dataset naming `boards_k / policies_k / values_k` and the six `game_stats`
counters (:181-208).  Games shard over ranks by index (game g -> rank g mod world); the search path has no
collective, finished trajectories are gathered to rank 0 (the single writer) with `torch.distributed`.
Randomness: tau sampling and the opening book use one numpy Generator per GLOBAL game id and the device Dirichlet
noise is keyed by the global game id, so a game's trajectory does not depend on the number of GPUs.
"""
import json
import os

import numpy as np

from . import games as G
from .engine import DIMS, Engine

try:  # the reference writes HDF5; h5py is not part of this image, so the same schema goes into an .npz otherwise
    import h5py as _h5
except Exception:  # noqa: BLE001
    _h5 = None


# ---------------------------------------------------------------------------------------------- replay writer --
_NPY_HEADERS = {}


def _npy_bytes(arr):
    """`arr` as the bytes of a .npy file (format 1.0); the header depends only on dtype and shape and is cached"""
    k = (arr.dtype.str, arr.shape)
    h = _NPY_HEADERS.get(k)
    if h is None:
        import io
        bio = io.BytesIO()
        np.lib.format.write_array_header_1_0(bio, np.lib.format.header_data_from_array_1_0(arr))
        h = _NPY_HEADERS[k] = bio.getvalue()
    return h + arr.tobytes()


class ReplayWriter:
    """`Self_Play_Data` with the reference schema (Self_Play.py:178-208): `game_stats` uint32[6] =
    [max game length, total positions, games, wins(-1), draws, wins(+1)] and per game and augmentation
    `boards_k` (T,H,W,C), `policies_k` (T,P) f32, `values_k` (T,1) f32.  HDF5 when h5py is importable, else
    `Self_Play_Data.npz` holding the same names.

    STREAMING: every game goes to the file when `add_game` is called (an .npz is a zip archive of .npy members, opened in
    append mode and written uncompressed), so the writer holds only `game_stats` and the dataset counter in memory - a
    generation of 131072 Gomoku games x 8 augmentations is ~50 GB of datasets.  `game_stats` is written by `flush()`;
    re-opening a finished archive to append more games (the resume rule of Self_Play.py:267-272) first copies its members,
    minus `game_stats`, into a fresh archive, because zip members cannot be replaced in place."""

    def __init__(self, folder_path):
        self.folder = folder_path
        os.makedirs(folder_path, exist_ok=True)
        self.h5_path = os.path.join(folder_path, "Self_Play_Data.h5")
        self.npz_path = os.path.join(folder_path, "Self_Play_Data.npz")
        self.use_h5 = _h5 is not None
        self.stats = np.zeros(6, dtype=np.uint32)
        self.n_datasets = 0          # (len(file.keys()) - 1) // 3 of the reference
        self._zip = None
        self.keys = ["game_stats"]   # creation order (what `file.keys()` lists in the reference's numbering rule)
        if not self.use_h5 and os.path.exists(self.npz_path):
            with np.load(self.npz_path) as z:
                self.stats = np.asarray(z["game_stats"], dtype=np.uint32).copy()
                names = [k for k in z.files if k != "game_stats"]
            self.n_datasets = len(names) // 3
            self.keys += names

    @property
    def data(self):
        """the archive's content as a dict (tests, small files): game_stats + every dataset, in creation order"""
        if self.use_h5:
            with _h5.File(self.h5_path, "r") as f:
                return {k: np.asarray(f[k]) for k in f.keys()}
        out = {"game_stats": self.stats.copy()}
        self._close_zip()
        if os.path.exists(self.npz_path):
            with np.load(self.npz_path) as z:
                for k in self.keys[1:]:
                    out[k] = z[k]
        return out

    def games_done(self):
        if self.use_h5:
            try:
                with _h5.File(self.h5_path, "r") as f:
                    return int(f["game_stats"][2]) if "game_stats" in f else 0
            except OSError:         # no file yet (h5py raises FileNotFoundError, an OSError)
                return 0
        return int(self.stats[2])

    def _open_zip(self):
        import zipfile
        if self._zip is not None:
            return self._zip
        if os.path.exists(self.npz_path):      # resume: carry the datasets over, drop the stale game_stats member
            tmp = self.npz_path + ".tmp"
            with zipfile.ZipFile(self.npz_path, "r") as src, zipfile.ZipFile(tmp, "w", zipfile.ZIP_STORED, allowZip64=True) as dst:
                for info in src.infolist():
                    if info.filename != "game_stats.npy":
                        with src.open(info) as fi, dst.open(info.filename, "w", force_zip64=True) as fo:
                            while True:
                                blk = fi.read(1 << 24)
                                if not blk:
                                    break
                                fo.write(blk)
            os.replace(tmp, self.npz_path)
            self._zip = zipfile.ZipFile(self.npz_path, "a", zipfile.ZIP_STORED, allowZip64=True)
        else:
            self._zip = zipfile.ZipFile(self.npz_path, "w", zipfile.ZIP_STORED, allowZip64=True)
        return self._zip

    def _close_zip(self):
        if self._zip is not None:
            self._zip.close()
            self._zip = None

    def add_game(self, boards_aug, policies_aug, values_aug, game_length, winner):
        """boards_aug (A,T,H,W,C), policies_aug (A,T,P), values_aug (A,T,1)"""
        if self.use_h5:
            with _h5.File(self.h5_path, "a") as f:
                if "game_stats" not in f:
                    f.create_dataset("game_stats", data=np.zeros(6, dtype=np.uint32))
                st = f["game_stats"]
                self._bump(st, boards_aug.shape[1], game_length, winner)
                k0 = (len(f.keys()) - 1) // 3
                for inc in range(policies_aug.shape[0]):
                    for name, arr, dt in self._triple(boards_aug, policies_aug, values_aug, inc):
                        f.create_dataset("%s_%d" % (name, k0 + inc), maxshape=(None, *arr.shape[1:]), dtype=dt, data=arr, chunks=None)
            return
        zf = self._open_zip()
        self._bump(self.stats, boards_aug.shape[1], game_length, winner)
        k0 = self.n_datasets
        for inc in range(policies_aug.shape[0]):
            for name, arr, dt in self._triple(boards_aug, policies_aug, values_aug, inc):
                key = "%s_%d" % (name, k0 + inc)
                zf.writestr(key + ".npy", _npy_bytes(np.ascontiguousarray(arr, dtype=dt)))   # one call per member: a generation
                self.keys.append(key)                                                          # of short games is bound by this loop
        self.n_datasets += policies_aug.shape[0]

    @staticmethod
    def _triple(boards_aug, policies_aug, values_aug, inc):
        return (("boards", boards_aug[inc], boards_aug.dtype), ("policies", policies_aug[inc], np.float32),
                ("values", values_aug[inc], np.float32))

    @staticmethod
    def _bump(st, n_positions, game_length, winner):
        if st[0] < game_length:
            st[0] = game_length
        st[1] += n_positions
        st[2] += 1
        st[winner + 4] += 1

    def flush(self):
        """finish the archive: `game_stats` is its last member; the writer can be re-opened to append later"""
        if self.use_h5:
            return
        zf = self._open_zip()
        with zf.open("game_stats.npy", "w") as fo:
            np.lib.format.write_array(fo, self.stats, allow_pickle=False)
        self._close_zip()


def game_values(q, z, winner):
    """Self_Play.py:159-172: z sign / draw rules, value = 0.5 * (z + q) -> (T, 1) float32"""
    q = np.asarray(q, dtype=np.float32).reshape((-1, 1))
    z = np.asarray(z, dtype=np.float32).reshape((-1, 1)).copy()
    if winner == z[-1][0] == -1:
        z *= -1.0
    elif winner == 0:
        z[:] = 0.0
    return 0.5 * (z + q)


def finalize_game(game_obj, states, policies, q, z, winner):
    """Self_Play.py:159-176 for one game on the host: targets + the game's own `augment_sample`."""
    states = np.asarray(states, dtype=game_obj.board.dtype)
    policies = np.asarray(policies, dtype=np.float32)
    values = game_values(q, z, winner)
    b_aug, p_aug = game_obj.augment_sample(states, policies)
    b_aug, p_aug = np.asarray(b_aug), np.asarray(p_aug)
    v_aug = np.repeat(np.expand_dims(values, 0), repeats=p_aug.shape[0], axis=0)
    return b_aug, p_aug, v_aug


def augmentation_tables(game_obj):
    """The game's `augment_sample` (Gomoku.py:264-303, Connect4.py:427-445, Tictactoe.py:322-358) as gather tables for
    `gaz_augment`: out[a][t][j] = in[t][perm[a][j]].  Derived by probing the game's OWN method with one-hot inputs, so a
    game plugin whose augmentation is a pure re-ordering needs no second implementation.  Returns (perm_state (A, S) int32,
    perm_policy (A, P) int32) or None when the method is not a permutation (the host path is used then)."""
    st0 = np.asarray(game_obj.get_input_state())
    S, P = int(st0.size), int(game_obj.policy_shape[0])
    T = max(S, P)
    states = np.zeros((T, S), dtype=game_obj.board.dtype)
    states[np.arange(S), np.arange(S)] = 1
    pols = np.zeros((T, P), dtype=np.float32)
    pols[np.arange(P), np.arange(P)] = 1.0
    b, p = game_obj.augment_sample(states.reshape((T,) + st0.shape), pols)
    b, p = np.asarray(b).reshape(-1, T, S), np.asarray(p).reshape(-1, T, P)
    A = b.shape[0]
    if p.shape[0] != A or np.any((b != 0).sum(1)[:, :] != 1) or np.any((p != 0).sum(1) != 1):
        return None
    perm_s = np.argmax(b != 0, axis=1).astype(np.int32)       # (A, S): which one-hot row lit output position j
    perm_p = np.argmax(p != 0, axis=1).astype(np.int32)
    if perm_s.max() >= S or perm_p.max() >= P:
        return None
    return perm_s, perm_p


def finalize_games(game_obj, games, device=0, lib=None, tables=None, chunk_positions=1 << 16):
    """Self_Play.py:159-176 for a LIST of finished games: targets on the host (a few flops per position), the 8-fold / 2-fold
    augmentation of every position as one table-driven gather per chunk on the device (`gaz_augment`).  Yields
    (game, boards_aug (A,T,H,W,C), policies_aug (A,T,P), values_aug (A,T,1)) in order - a generator, so a streaming writer
    never holds more than one chunk."""
    import ctypes as C
    from . import _lib
    lib = lib if lib is not None else _lib.load()
    tables = tables if tables is not None else augmentation_tables(game_obj)
    st_shape = np.asarray(game_obj.get_input_state()).shape
    bdt = game_obj.board.dtype
    if tables is None or bdt != np.int8:
        for g in games:      # a game whose augmentation is not a re-ordering (or whose boards are not int8): host path
            yield (g,) + finalize_game(game_obj, g["states"], g["policies"], g["q"], g["z"], g["winner"])
        return
    perm_s, perm_p = tables
    A, S, P = perm_s.shape[0], perm_s.shape[1], perm_p.shape[1]
    i = 0
    while i < len(games):
        j, npos = i, 0
        while j < len(games) and (j == i or npos + games[j]["length"] <= chunk_positions):
            npos += games[j]["length"]
            j += 1
        st = np.ascontiguousarray(np.concatenate([np.asarray(g["states"], dtype=np.int8).reshape(g["length"], S) for g in games[i:j]]))
        po = np.ascontiguousarray(np.concatenate([np.asarray(g["policies"], dtype=np.float32).reshape(g["length"], P) for g in games[i:j]]))
        so = np.empty((A, npos, S), np.int8)
        pout = np.empty((A, npos, P), np.float32)
        rc = lib.gaz_augment(int(device), st.ctypes.data_as(C.c_void_p), po.ctypes.data_as(C.c_void_p), npos, S, P,
                             perm_s.ctypes.data_as(C.c_void_p), perm_p.ctypes.data_as(C.c_void_p), A,
                             so.ctypes.data_as(C.c_void_p), pout.ctypes.data_as(C.c_void_p))
        if rc < 0:
            raise RuntimeError(lib.gaz_last_error().decode())
        off = 0
        for g in games[i:j]:
            T = g["length"]
            values = game_values(g["q"], g["z"], g["winner"])
            yield (g, so[:, off:off + T].reshape((A, T) + st_shape), pout[:, off:off + T],
                   np.repeat(np.expand_dims(values, 0), repeats=A, axis=0))
            off += T
        i = j


# ---------------------------------------------------------------------------------------- the batched driver --
def match_tree_nets(game_ids):
    """Network of each PUCT tree in a match, uint8 (len(game_ids), 2): tree k of the game with global id g searches with
    network (k + g) % 2.  Tree 0 plays player -1, who moves first from the empty board, so network 0 moves first in the
    even games and network 1 in the odd ones."""
    g = np.asarray(game_ids, dtype=np.int64).reshape(-1, 1)
    return ((g + np.arange(2)) % 2).astype(np.uint8)


class BatchedSelfPlay:
    """Plays the games `game_ids` (global ids) on one device, `n_slots` at a time.

    Matches and tournaments (arena.play_match / arena.play_tournament): `opponents = [(spec_k, weights_k), ...]` attaches
    networks 1..K-1 (K <= 8; network 0 is `spec` / `weights`), and `tree_nets(game_id) -> (network of tree 0, network of
    tree 1)` says which network each of a game's two PUCT trees searches with.  `opponent = (spec_b, weights_b)` is
    `opponents = [opponent]` with `tree_nets` = match_tree_nets.  Networks of equal specs share one activation workspace
    (net.Net(share=...)).  `openings(game_id) -> (board, next_player, action id history)` seats that position instead of
    the empty board; `limits` are the K per-network iteration limits (default `self.limit` for every network).  The finished
    records of a match also hold the played action ids and the iterations of every search.  `train_config["eval_symmetry"]`
    ("none" by default: the reference's evaluation; "random" or "ensemble", seeded from `seed`) is how every network evaluates
    (Engine.set_eval_symmetry)."""

    def __init__(self, game_class, build_config, train_config, game_ids, n_slots, device=0, evaluator="net",
                 spec=None, weights=None, seed=0, lib=None, hash_salt=0, node_cap=None, slot_cap=None,
                 use_noise=True, slot_pool_fraction=None, opponent=None, openings=None, limits=None, opponents=None,
                 tree_nets=None):
        self.game_class = game_class
        self.proto = game_class()
        self.name = G.game_name_of(self.proto)
        self.H, self.W, self.C, self.P = DIMS[self.name]
        self.tc, self.bc = train_config, build_config
        self.gumbel = bool(train_config.get("use_gumbel", False))
        self.tpg = 1 if self.gumbel else 2
        self.queue = list(game_ids)
        self.n_slots = max(1, min(n_slots, len(self.queue))) if self.queue else 1
        self.seed = seed
        self.evaluator = evaluator
        self.hash_salt = hash_salt
        limit = train_config["MCTS_iteration_limit"]
        self.limit = int(limit) if self.gumbel else int(limit * 1.5)          # Self_Play.py:99
        if opponent is not None:
            if opponents is not None:
                raise ValueError("pass either opponent or opponents")
            opponents, tree_nets = [opponent], None
        self.opponents = [] if opponents is None else list(opponents)
        self.n_nets = 1 + len(self.opponents)
        self.match = self.n_nets > 1
        if self.n_nets > 8:
            raise ValueError("at most 8 networks, got %d" % self.n_nets)
        if self.match and self.gumbel:
            raise ValueError("a match needs two PUCT trees per game (one per network); use_gumbel runs one tree per game")
        if self.match and evaluator != "net":
            raise ValueError("a match needs evaluator='net'")
        if tree_nets is None and self.n_nets > 2:
            raise ValueError("%d networks need tree_nets(game_id)" % self.n_nets)
        self.tree_nets_of = tree_nets          # None: match_tree_nets
        self.openings = openings
        if limits is not None and len(limits) != self.n_nets:
            raise ValueError("limits: %d values for %d networks" % (len(limits), self.n_nets))
        self.limits = None if limits is None else tuple(int(x) for x in limits)
        self.tree_net = np.zeros((self.n_slots, self.tpg), np.uint8)   # network of every tree (all 0 outside a match)
        search_limit = self.limit if self.limits is None else max(self.limits)
        self.max_actions = int(train_config["max_actions"])
        stablemax = bool(build_config.get("use_stablemax"))
        L = 7 if self.name == "connect4" else self.P
        # iterations a PUCT run can really make: `iteration_limit < n_legal -> 3 * n_legal` (MCTS.py:543-546)
        self.eff_limit = search_limit if (self.gumbel or search_limit >= L) else 3 * L
        if node_cap is None:
            # Pools are sized for the tail of WHOLE games, not for the opening: an expansion whose position has terminal
            # replies creates a terminal parent and its k terminal children (MCTS.py:367-428), and the sub-tree kept
            # from the previous move comes on top of the limit new nodes.  Measured peaks per tree (emulated engine, 12
            # full Gomoku games at 1200 iterations: 2806 nodes / 374 k child slots; a 4096-game Connect4 generation
            # overflowed 3.5 x limit nodes).  Gomoku: 4 x limit nodes (~100 B each) and 2 x limit x L child slots (5 B
            # each; only evaluated nodes own L slots) = 3.3 MB per tree; Connect4 / TicTacToe nodes are < 100 B all in.
            node_cap = (4 if self.name == "gomoku" else 8) * self.eff_limit + 4 * L + 64
            if slot_cap is None and self.name == "gomoku" and not self.gumbel:
                slot_cap = 2 * self.eff_limit * L + 256
            if self.gumbel:
                node_cap = int(self.limit * 1.5) + 2 * L + 64
            slot_cap = node_cap * min(L, 225) + 256 if slot_cap is None else slot_cap
        # child slots come from an engine-wide page pool; train_config["slot_pool_fraction"] (< 1) sizes it from the mean tree
        # occupancy instead of the per-tree worst case, so more games fit a GPU (see _relieve_full_pools for the back-stop)
        frac = slot_pool_fraction if slot_pool_fraction is not None else float(train_config.get("slot_pool_fraction", 1.0))
        slot_pool = 0 if frac >= 1.0 else int(frac * self.n_slots * self.tpg * slot_cap)
        self.eng = Engine(self.name, n_games=self.n_slots, mode="gumbel" if self.gumbel else "puct",
                          trees_per_game=self.tpg, node_cap=node_cap, slot_cap=slot_cap, slot_pool=slot_pool,
                          c_puct_init=float(train_config.get("c_puct_init", 2.5)), m=int(train_config.get("m", 16)),
                          c_visit=float(train_config.get("c_visit", 50.0)), c_scale=float(train_config.get("c_scale", 1.0)),
                          activation_fn="stablemax" if stablemax else "softmax", device=device, lib=lib)
        # train_config["eval_cache_entries"] > 0: device-side evaluation cache (what max_cache_depth / Session_Cache.Cache_Wrapper
        # are to the reference, Self_Play.py:233-235); "eval_cache_shared": one table for all games instead of per-game entries
        if int(train_config.get("eval_cache_entries", 0) or 0) > 0:
            self.eng.enable_eval_cache(int(train_config["eval_cache_entries"]), shared=bool(train_config.get("eval_cache_shared", False)))
        self.nets = []
        if evaluator == "net":
            from .net import Net
            for sp_k, w_k in [(spec, weights)] + self.opponents:
                donor = next((n for n in self.nets if n.spec == sp_k), None)    # attached networks run one after another
                # larger request lists are served in chunks
                self.nets.append(Net(sp_k, w_k, max_batch=self.n_slots, device=device, share=donor))
            if self.match:
                self.eng.attach_nets(self.nets)
            else:
                self.nets[0].attach(self.eng)
        self.net = self.nets[0] if self.nets else None
        # train_config["eval_symmetry"]: "none" (default, the reference's evaluation), "random" (each request under one board
        # symmetry drawn from a hash of the seed, the game's global id and the position) or "ensemble" (the mean over all
        # symmetries, n times the network work); only "none" keeps reference parity (Engine.set_eval_symmetry)
        sym = str(train_config.get("eval_symmetry", "none") or "none")
        if sym != "none":
            if evaluator != "net":
                raise ValueError("eval_symmetry=%r needs evaluator='net'" % sym)
            self.eng.set_eval_symmetry(sym, seed)
        if not self.gumbel and use_noise:
            self.eng.set_noise(float(train_config.get("dirichlet_alpha", 0.3)), 0.25, seed)   # Self_Play.py:38-46
        self.use_gumbel_noise = self.gumbel and use_noise
        # per-slot host state
        self.slot_game = np.full(self.n_slots, -1, np.int64)      # global game id or -1 (idle)
        self.rngs = [None] * self.n_slots
        self.traj = [None] * self.n_slots
        self.finished = []
        self.pool_rebuilds = 0    # trees given a fresh root because their pool could not hold another move (see _relieve_full_pools)
        self.sims = 0
        self.moves = 0

    # ---- evaluator plumbing --------------------------------------------------------------------------------
    def _serve(self, n):
        if n > 0:
            if self.evaluator == "net":
                self.eng.eval_net()
            else:
                self.eng.eval_hash(self.hash_salt, self.gumbel)
        self.eng.expand()

    def _rounds(self, n):
        if self.evaluator == "net":
            self.eng.rounds_net(n)
        else:
            self.eng.rounds_hash(n, self.hash_salt, self.gumbel)

    # ---- slots ---------------------------------------------------------------------------------------------
    def _seat(self, slots):
        """put queued games into `slots` (empty boards, fresh roots)"""
        seated = []
        for s in slots:
            if not self.queue:
                self.slot_game[s] = -1
                continue
            gid = self.queue.pop(0)
            self.slot_game[s] = gid
            self.rngs[s] = np.random.Generator(np.random.PCG64([self.seed, int(gid)]))
            self.traj[s] = dict(states=[], policies=[], q=[], z=[], actions=[], iterations=[])
            if self.openings is None:
                self.eng.set_game(int(s), np.zeros((self.H, self.W), np.int8), -1, [])
            else:
                board, next_player, history = self.openings(int(gid))
                self.eng.set_game(int(s), board, next_player, list(history))
            seated.append(s)
        keys = np.repeat(np.where(self.slot_game >= 0, self.slot_game, 0).astype(np.uint64), self.tpg)
        self.eng.set_tree_keys(keys * np.uint64(2) + np.tile(np.arange(self.tpg, dtype=np.uint64), self.n_slots))
        if self.match:   # before the new roots below are evaluated
            if self.tree_nets_of is None:
                self.tree_net = match_tree_nets(np.where(self.slot_game >= 0, self.slot_game, 0))
            else:        # idle slots search nothing; their trees stay on network 0
                self.tree_net = np.array([self.tree_nets_of(int(g)) if g >= 0 else (0, 0) for g in self.slot_game],
                                         np.uint8).reshape(self.n_slots, 2)
            self.eng.set_tree_nets(self.tree_net.reshape(-1))
        if seated:
            mask = np.zeros((self.n_slots, self.tpg), np.uint8)
            mask[seated] = 1
            for k in range(self.tpg):   # one tree per game at a time keeps the evaluation batch <= n_slots
                m = np.zeros_like(mask)
                m[:, k] = mask[:, k]
                self._serve(self.eng.new_roots(m.reshape(-1)))

    def live(self):
        return self.slot_game >= 0

    def _relieve_full_pools(self, cont, next_mover):
        """The reference's trees are unbounded Python objects; ours live in fixed per-tree pools.  A kept sub-tree grows
        with the concentration of the search (steady state ~ limit / (1 - share of the played line)), so no static size is
        safe for every network.  After re-rooting, a tree that is about to search and could not hold one more move's worth
        (2 nodes per iteration, L child slots per evaluated node) gets a fresh root instead - what `prune_tree` does for an
        unseen action (MCTS.py:661-671): one evaluation, no reuse for that move.  Counted in `pool_rebuilds`."""
        e = self.eng
        sizes = e.tree_sizes().reshape(self.n_slots, self.tpg, 2)
        nxt = (np.asarray(next_mover) > 0).astype(np.int64)                 # the tree of the side to move runs next
        mine = sizes[np.arange(self.n_slots), nxt]
        L = 7 if self.name == "connect4" else self.P
        full = cont & ((mine[:, 0] + 2 * self.eff_limit > e.node_cap) | (mine[:, 1] + self.eff_limit * L > e.slot_cap))
        # shared page pool: the trees about to search must be able to take the pages one more move can need; if the pool is
        # short the LARGEST kept sub-trees give theirs back (fresh root, counted)
        pinfo = e.pool_info()
        if pinfo["pages"] < e.n_trees * pinfo["max_pages_per_tree"]:
            ps = pinfo["page_slots"]
            demand = np.where(cont & ~full, -(-(mine[:, 1] + self.eff_limit * L) // ps) - (-(-mine[:, 1] // ps)), 0)
            short = int(demand.sum()) - pinfo["free"]
            for s in np.argsort(-mine[:, 1]):
                if short <= 0:
                    break
                if cont[s] and not full[s]:
                    full[s] = True
                    short -= int(demand[s]) + int(-(-mine[s, 1] // ps)) - 1
        if not full.any():
            return
        mask = np.zeros((self.n_slots, self.tpg), np.uint8)
        mask[np.nonzero(full)[0], nxt[full]] = 1
        self.pool_rebuilds += int(full.sum())
        self._serve(e.new_roots(mask.reshape(-1)))

    # ---- one move of every live game -------------------------------------------------------------------
    def step(self):
        e = self.eng
        live = self.live()
        if not live.any():
            return False
        states, ginfo = e.get_states()
        mover = ginfo[:, 0]
        hist_len = ginfo[:, 1]
        run_tree = np.zeros(self.n_slots, np.int64) if self.gumbel else (mover > 0).astype(np.int64)
        limits = np.zeros((self.n_slots, self.tpg), np.int32)
        run_limit = self.limit if self.limits is None else \
            np.asarray(self.limits, np.int32)[self.tree_net[np.arange(self.n_slots), run_tree]]
        limits[np.arange(self.n_slots), run_tree] = np.where(live, run_limit, 0)
        if self.use_gumbel_noise:   # MCTS_Gumbel.py:592-594: Gumbel(0,1) on the root logits, one stream per game
            noise = np.zeros((self.n_slots, 256), np.float64)
            for s in np.nonzero(live)[0]:
                noise[s] = self.rngs[s].gumbel(size=256)
            e.set_gumbel_noise(noise)
        e.run_begin(limits.reshape(-1))
        while e.remaining() > 0:
            self._rounds(32)
        vis, val, tinfo = e.root_dense(want_values=True)
        vis = vis.reshape(self.n_slots, self.tpg, self.P)[np.arange(self.n_slots), run_tree]
        val = val.reshape(self.n_slots, self.tpg, self.P)[np.arange(self.n_slots), run_tree]
        tinfo = tinfo.reshape(self.n_slots, self.tpg, 4)[np.arange(self.n_slots), run_tree]
        self.sims += int(tinfo[live, 2].sum())
        if self.gumbel:
            pi = e.gumbel_pi_dense().reshape(self.n_slots, self.P)
        actions = np.full(self.n_slots, -1, np.int16)
        for s in np.nonzero(live)[0]:
            v = vis[s].astype(np.float64)
            if self.gumbel:
                policy = pi[s]
                a = int(tinfo[s, 1])
                with np.errstate(divide="ignore", invalid="ignore"):
                    q = val[s, a] / vis[s, a] if vis[s, a] > 0 else pi[s, a]     # MCTS_Gumbel.py:648-666
            else:
                policy = (v / v.sum()).astype(np.float32)
                move_no = int(hist_len[s])
                first = move_no % 2 == 0
                explore = (move_no // 2 < self.tc.get("num_explore_actions_first", 0)) if first else \
                    ((move_no + 1) // 2 < self.tc.get("num_explore_actions_second", 0))       # Self_Play.py:87-95
                if explore:  # tau = 1: weights visits / root.visits, renormalised (MCTS.py:605-610)
                    w = v / float(tinfo[s, 0]) if tinfo[s, 0] > 0 else v
                    w = w / w.sum()
                    a = int(self.rngs[s].choice(self.P, p=w))
                else:
                    a = int(tinfo[s, 1])
                q = np.float32(val[s, a]) / np.float32(vis[s, a]) if vis[s, a] > 0 else np.float32(0.0)
            t = self.traj[s]
            t["states"].append(states[s].copy())
            t["policies"].append(policy)
            t["q"].append(np.float32(q))
            t["z"].append(float(mover[s]))
            t["iterations"].append(int(tinfo[s, 2]))
            if hist_len[s] == 0 and self.tc.get("opening_actions", False):               # Self_Play.py:130-140
                acts, weights = zip(*self.tc["opening_actions"])
                acts = [G.action_to_id(self.name, x) for x in acts]
                weights = list(weights)
                if sum(weights) < 1.0:
                    acts.append(a)
                    weights.append(1.0 - sum(weights))
                a = int(acts[int(self.rngs[s].choice(len(acts), p=np.asarray(weights) / sum(weights)))])
            actions[s] = a
            t["actions"].append(a)
        winners = e.apply_actions(actions)
        self.moves += int(live.sum())
        done = []
        for s in np.nonzero(live)[0]:
            w = int(winners[s])
            n_act = int(hist_len[s]) + 1      # plies of the game, an opening seated by `openings` included
            if n_act >= self.max_actions:
                w = 0      # Self_Play.py:155-157: `if actions_count == max_actions: winner = 0` - a WIN on that ply is a draw too
            if w != -2:
                done.append((s, w))
        done_slots = [s for s, _ in done]
        cont = live.copy()
        cont[done_slots] = False
        pa = np.repeat(np.where(cont, actions, -1).astype(np.int16), self.tpg)
        create_new = True if self.gumbel else bool(self.tc.get("create_new_root", False))
        self._serve(e.prune(pa, create_new_root=create_new))
        if not create_new:
            self._relieve_full_pools(cont, -mover)
        for s, w in done:
            t = self.traj[s]
            rec = dict(game_id=int(self.slot_game[s]), winner=w, length=len(t["z"]),
                       states=np.asarray(t["states"], dtype=np.int8),
                       policies=np.asarray(t["policies"], dtype=np.float32),
                       q=np.asarray(t["q"], dtype=np.float32), z=np.asarray(t["z"], dtype=np.float32))
            if self.match:
                rec.update(actions=np.asarray(t["actions"], dtype=np.int16), iterations=np.asarray(t["iterations"], dtype=np.int32))
            self.finished.append(rec)
            self.traj[s] = None
        if done_slots:
            self._seat(done_slots)
        return True

    def play(self, progress=None):
        self._seat(list(range(self.n_slots)))
        while self.step():
            st = self.eng.status()      # checked after every move: a tree pool that overflowed stops growing, so the
            if st != 0:                 # searches would silently differ from the reference's - fail before more is played
                raise RuntimeError("engine status %d (1 node overflow, 2 slot overflow): raise node_cap / slot_cap" % st)
            if progress is not None:
                progress(self)
        return self.finished

    def close(self):
        self.eng.close()
        for n in self.nets:
            n.close()


# ------------------------------------------------------------------------------------------- trajectory gather --
def pack_games(finished):
    """list of finished-game dicts -> one uint8 buffer (JSON index + raw arrays)"""
    index, blobs, off = [], [], 0
    for g in finished:
        rec = dict(game_id=g["game_id"], winner=g["winner"], length=g["length"], arrays={})
        for k in ("states", "policies", "q", "z"):
            a = np.ascontiguousarray(g[k])
            rec["arrays"][k] = dict(dtype=str(a.dtype), shape=list(a.shape), offset=off, nbytes=a.nbytes)
            blobs.append(a.reshape(-1).view(np.uint8))
            off += a.nbytes
        index.append(rec)
    head = np.frombuffer(json.dumps(index).encode(), dtype=np.uint8)
    body = np.concatenate(blobs) if blobs else np.zeros(0, np.uint8)
    return np.concatenate([np.array([len(head)], dtype=np.int64).view(np.uint8), head, body])


def unpack_games(buf):
    buf = np.asarray(buf, dtype=np.uint8)
    n = int(buf[:8].view(np.int64)[0])
    index = json.loads(bytes(buf[8:8 + n]).decode())
    body = buf[8 + n:]
    out = []
    for rec in index:
        g = dict(game_id=rec["game_id"], winner=rec["winner"], length=rec["length"])
        for k, a in rec["arrays"].items():
            g[k] = body[a["offset"]:a["offset"] + a["nbytes"]].view(np.dtype(a["dtype"])).reshape(a["shape"]).copy()
        out.append(g)
    return out


def gather_games(finished, device=None, stats=None):
    """All ranks -> rank 0: lengths by all_gather, then one padded byte buffer per rank by gather (NCCL over NVLink when
    the process group is NCCL and `device` is a CUDA device, gloo on CPU).  Returns the merged list on rank 0, [] elsewhere."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return sorted(finished, key=lambda g: g["game_id"])
    import time
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cpu") if device is None else torch.device(device)
    buf = torch.from_numpy(pack_games(finished).copy()).to(dev)
    # the first gather on a process group builds its point-to-point channels (~0.1 s): a one-byte gather takes that hit so
    # that `collective_s` times the payload exchange
    warm = torch.zeros(1, dtype=torch.uint8, device=dev)
    dist.gather(warm, gather_list=[torch.zeros(1, dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None, dst=0)
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    size = torch.tensor([buf.numel()], dtype=torch.int64, device=dev)
    sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(sizes, size)
    mx = int(max(int(s.item()) for s in sizes))
    padded = torch.zeros(mx, dtype=torch.uint8, device=dev)
    padded[:buf.numel()] = buf
    outs = [torch.zeros(mx, dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None
    dist.gather(padded, gather_list=outs, dst=0)
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    if stats is not None:    # the collective alone (all_gather of sizes + padded gather), and the payload this rank sent
        stats.update(collective_s=time.perf_counter() - t0, bytes=int(buf.numel()), padded_bytes=mx)
    if rank != 0:
        return []
    merged = []
    for r in range(world):
        merged += unpack_games(outs[r][:int(sizes[r].item())].cpu().numpy())
    merged.sort(key=lambda g: g["game_id"])
    return merged


# ------------------------------------------------------------------------------------------------ entry point --
def net_spec_from_configs(game_name, build_config, train_config):
    from . import netspec
    gumbel = bool(train_config.get("use_gumbel", False))
    head = "linear" if gumbel else ("stablemax" if build_config.get("use_stablemax") else "softmax")
    over = {}
    if "num_resnet_layers" in build_config:
        over["num_blocks"] = int(build_config["num_resnet_layers"])
    if "num_filters" in build_config and game_name != "tictactoe":   # TicTacToe/Build_Model.py:22 hard-codes ResNet_Block(64)
        over["filters"] = int(build_config["num_filters"])
    # Squeeze-Excitation is opt-in: the reference's builders never wire SE_Block in (Net/ResNet/ResNet_Block.py:27-41) and
    # its build_config has no such key, so the reference's own configs must give the reference's architecture (and a
    # keras_bridge checkpoint must load); BASELINE configs[2] asks for it explicitly with use_se=True
    over["use_se"] = bool(build_config.get("use_se", False))
    return netspec.build_spec(game_name, head, **over)


def run_self_play(game_class, configs, folder_path, per_process_wait_time=1e-3, weights=None, seed=None, evaluator="net",
                  lib=None, timings=None):
    """Same call as the reference's `run_self_play(game_class, configs, folder_path, per_process_wait_time)`; plays
    `games_per_generation - game_stats[2]` games (resume rule of Self_Play.py:267-272) on this rank's share of the
    game ids and appends them to `folder_path/Self_Play_Data` on rank 0.  Extra keys read from train_config:
    `games_per_gpu` (concurrent games per GPU, default 4096) and `eval_symmetry` ("none", the default and the reference's
    evaluation; "random" or "ensemble", see BatchedSelfPlay - seeded from `seed`, and not reference parity).  `weights`: Keras-layout dict or a checkpoint path
    (default `folder_path/model.npz`, else random init).  `seed`: None draws one from the OS on rank 0 (the reference
    reseeds every worker from entropy, Self_Play.py:221) and broadcasts it; an explicit seed makes a run reproducible.
    `evaluator`: "net" (CUDA network), "hash" (deterministic parity evaluator) or "random" - a uniform-random policy /
    value per position, what the reference plays generation 0 with (session=None, MCTS.py:236-240).
    `timings`: optional dict that receives wall-clock seconds per phase and the bytes gathered."""
    import time
    build_config, train_config = configs[0], configs[1]
    rank, world, device = 0, 1, 0
    dist = None
    try:
        import torch.distributed as dist_mod
        if dist_mod.is_available() and dist_mod.is_initialized():
            dist = dist_mod
            rank, world = dist.get_rank(), dist.get_world_size()
            device = int(os.environ.get("LOCAL_RANK", rank))
    except Exception:  # noqa: BLE001
        dist = None

    def bcast_int(v):
        if world == 1:
            return int(v)
        import torch
        t = torch.tensor([int(v)], dtype=torch.int64)
        if dist.get_backend() == "nccl":
            t = t.cuda(device)
        dist.broadcast(t, src=0)
        return int(t.item())

    writer = ReplayWriter(folder_path) if rank == 0 else None
    done = bcast_int(writer.games_done() if rank == 0 else 0)
    if seed is None:
        seed = int.from_bytes(os.urandom(4), "little") if rank == 0 else 0
    seed = bcast_int(seed)
    games_left = int(train_config["games_per_generation"]) - done
    if games_left <= 0:
        print(f"Finished generating {train_config['games_per_generation']} games!")
        return []
    ids = [g for g in range(done, done + games_left) if g % world == rank]
    spec = w = None
    name = G.game_name_of(game_class())
    if evaluator == "net":
        from . import netspec, session
        if isinstance(weights, str) or (weights is None and os.path.exists(os.path.join(folder_path, "model.npz"))):
            spec, w = session.load_checkpoint(weights if isinstance(weights, str) else os.path.join(folder_path, "model.npz"))
        else:
            spec = net_spec_from_configs(name, build_config, train_config)
            w = weights if weights is not None else netspec.init_weights(spec, seed=seed)
    t0 = time.perf_counter()
    sp = BatchedSelfPlay(game_class, build_config, train_config, ids, int(train_config.get("games_per_gpu", 4096)),
                         device=device, evaluator="hash" if evaluator == "random" else evaluator, spec=spec, weights=w, seed=seed,
                         lib=lib, hash_salt=seed if evaluator == "random" else 0)
    finished = sp.play()
    if sp.pool_rebuilds:
        print("run_self_play: %d tree(s) restarted from a fresh root because their pool could not hold another move "
              "(raise node_cap / slot_cap to keep the sub-tree reuse)" % sp.pool_rebuilds)
    sims, moves = sp.sims, sp.moves
    sp.close()
    t1 = time.perf_counter()
    dev = None
    if world > 1:
        dev = ("cuda:%d" % device) if dist.get_backend() == "nccl" else None
    stats = {}
    merged = gather_games(finished, device=dev, stats=stats)
    t2 = time.perf_counter()
    if rank == 0:
        proto = game_class()
        for g, b, p, v in finalize_games(proto, merged, device=device, lib=lib):
            writer.add_game(b, p, v, g["length"], g["winner"])
        writer.flush()
    t3 = time.perf_counter()
    if timings is not None:
        timings.update(play_s=t1 - t0, gather_s=t2 - t1, write_s=t3 - t2, sims=int(sims), moves=int(moves), seed=int(seed),
                       gather_bytes=int(stats.get("bytes", 0)), gather_collective_s=float(stats.get("collective_s", 0.0)))
    return merged
