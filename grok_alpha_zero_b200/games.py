"""Game plugins with the reference's game-class interface (Guide.py:79-284).

Host-side mirrors of Gomoku/Gomoku.py:87-303, Connect4/Connect4.py:218-445 and TicTacToe/Tictactoe.py:130-358:
same attributes (`board`, `next_player`, `action_history`, `policy_shape`), same methods and the same static
`*_MCTS` functions with the same argument order, dtypes, action formats and quirks, so `Self_Play.py`,
`Game_Tester.py` and user scripts can use them unchanged.  The search itself never calls these per simulation -
rules, terminal look-ahead and input encoding run on the GPU as bitboard code (csrc/gaz_core.cuh) - they are
the API surface around it (live game object, post-game augmentation) and the CPU-side check of the device code.

Numeric note: the reference's numba `np.sum` is a left-to-right float32 sum (SURVEY V2); `_seq_sum` reproduces
it so that `get_legal_actions_policy_MCTS` is bit-identical.
"""
import numpy as np


def _seq_sum(v):
    """left-to-right float32 sum (what numba's np.sum does on a float32 vector)"""
    if len(v) == 0:
        return np.float32(0.0)
    return np.add.accumulate(np.asarray(v, dtype=np.float32), dtype=np.float32)[-1]


def _dihedral8(a):
    """[a, flipud, fliplr, rot90, flipud(rot90), fliplr(rot90), rot180, rot270] on the first two axes
    (Gomoku.py:264-297, Tictactoe.py:322-351)"""
    r1 = np.rot90(a, 1)
    return [a, np.flipud(a), np.fliplr(a), r1, np.flipud(r1), np.fliplr(r1), np.rot90(a, 2), np.rot90(a, 3)]


class _GridGame:
    """Shared behaviour of the two (x, y)-action games (Gomoku, TicTacToe)."""
    H = W = 0
    ACTION_DTYPE = np.int64

    def get_next_player(self):
        return self.next_player

    def get_legal_actions(self):
        return self.get_legal_actions_MCTS(self.board, -self.next_player,
                                           np.array(self.action_history, dtype=self.ACTION_DTYPE))

    def get_input_state(self):
        return self.get_input_state_MCTS(self.board, -self.next_player,
                                         np.array(self.action_history, dtype=self.ACTION_DTYPE))

    def compute_policy_improvement(self, statistics):
        new_policy = np.zeros((self.H, self.W), dtype=np.float32)
        for (x, y), prob in statistics:
            new_policy[y][x] = prob
        return new_policy.reshape(-1)

    def augment_sample(self, input_states, policies):
        """8 dihedral copies: boards (8, T, H, W, C) in the board dtype, policies (8, T, P) float32."""
        input_states = np.asarray(input_states)
        pol = np.asarray(policies, dtype=np.float32).reshape((-1, self.H, self.W))
        T = input_states.shape[0]
        boards = np.empty((8, T) + input_states.shape[1:], dtype=self.board.dtype)
        pols = np.empty((8, T, self.H * self.W), dtype=np.float32)
        for t in range(T):
            for k, (s, p) in enumerate(zip(_dihedral8(input_states[t]), _dihedral8(pol[t]))):
                boards[k, t] = s
                pols[k, t] = p.reshape(-1)
        return boards, pols


class Gomoku(_GridGame):
    """15x15 five-in-a-row, actions = (x, y) uint8 pairs (Gomoku/Gomoku.py:87-303)."""
    H = W = 15
    ACTION_DTYPE = np.uint8

    def __init__(self, width=15, height=15):
        self.board = np.zeros((height, width), dtype=np.int8)
        self.next_player = -1
        self.action_history = []
        self.policy_shape = (225,)

    def input_action(self):
        while True:
            try:
                coords = np.array(list(map(int, input("Action:").split(" "))))
                if self.board[coords[1]][coords[0]] == 0:
                    return coords
                print("Illegal move")
            except Exception:
                print("Invalid input")

    @staticmethod
    def get_legal_actions_MCTS(board, current_player, action_history):
        return np.argwhere(board == 0)[:, ::-1].astype(np.uint8)

    @staticmethod
    def get_legal_actions_policy_MCTS(board, current_player, action_history, policy, normalize=True, shuffle=False):
        empty = board.reshape(-1) == 0
        policy = policy[empty]
        if normalize:
            policy = policy / _seq_sum(policy)
        legal_actions = np.argwhere(board == 0)[:, ::-1].astype(np.uint8)
        if shuffle:
            idx = np.random.permutation(len(legal_actions))
            legal_actions, policy = legal_actions[idx], policy[idx]
        return legal_actions, policy

    def do_action(self, action):
        x, y = action
        assert self.board[y][x] == 0
        self.board[y][x] = self.next_player
        self.next_player *= -1
        self.action_history.append(np.array(action, dtype=np.uint8))

    @staticmethod
    def do_action_MCTS(board, action, next_player):
        x, y = action
        board[y][x] = next_player
        return board

    @staticmethod
    def get_input_state_MCTS(board, current_player, action_history):
        side = np.ones_like(board) * np.int8(-current_player)   # plane 0 = side to move
        return np.stack((side, board), -1)

    def check_win(self):
        return self.check_win_MCTS(self.board, -self.next_player, np.array(self.action_history, dtype=np.uint8))

    @staticmethod
    def check_win_MCTS(board, current_player, action_history):
        """>= 5 in a row through the LAST move; cells outside the board are skipped without resetting the run;
        no draw detection: a full board without a five returns -2 (Gomoku.py:192-255)."""
        cx, cy = int(action_history[-1][0]), int(action_history[-1][1])
        for dx, dy in ((1, 0), (0, 1), (1, 1), (-1, 1)):
            run = 0
            for i in range(-4, 5):
                x, y = cx + dx * i, cy + dy * i
                if 0 <= x <= 14 and 0 <= y <= 14:
                    if board[y][x] == current_player:
                        run += 1
                        if run == 5:
                            return current_player
                    else:
                        run = 0
        return -2


class TicTacToe(_GridGame):
    """3x3, actions = (x, y) pairs (TicTacToe/Tictactoe.py:130-358)."""
    H = W = 3
    ACTION_DTYPE = np.int64

    def __init__(self):
        self.board = np.zeros((3, 3), dtype=np.int8)
        self.next_player = -1
        self.action_history = []
        self.policy_shape = (9,)

    def input_action(self):
        while True:
            try:
                coords = input("Move:").split(" ")
                x, y = int(coords[0]), int(coords[1])
                if not (0 <= x <= 2 and 0 <= y <= 2) or self.board[y][x] != 0:
                    print("Illegal move given")
                    continue
                return [x, y]
            except Exception:
                print("Invalid Move")

    def get_legal_actions(self):
        return self.get_legal_actions_MCTS(self.board, -self.next_player, np.array(self.action_history))

    def get_input_state(self):
        return self.get_input_state_MCTS(self.board, -self.next_player, np.array(self.action_history))

    @staticmethod
    def get_legal_actions_MCTS(board, current_player, action_history):
        return np.argwhere(board == 0)[:, ::-1]

    @staticmethod
    def get_legal_actions_policy_MCTS(board, current_player, action_history, policy, normalize=True, shuffle=False):
        legal_actions = np.argwhere(board == 0)[:, ::-1]
        legal_policy = policy[board.reshape(-1) == 0]
        if normalize:
            legal_policy = legal_policy / _seq_sum(legal_policy)
        if shuffle:
            idx = np.random.permutation(len(legal_actions))
            legal_actions, legal_policy = legal_actions[idx], legal_policy[idx]
        return legal_actions, legal_policy

    def do_action(self, action):
        x, y = action
        if self.board[y][x] != 0:
            raise ValueError("Illegal move")
        self.board[y][x] = self.next_player
        self.next_player = self.next_player * -1
        self.action_history.append(action)

    @staticmethod
    def do_action_MCTS(board, action, next_player):
        x, y = action
        board[y][x] = next_player
        return board

    @staticmethod
    def get_input_state_MCTS(board, current_player, action_history):
        side = np.expand_dims(np.ones_like(board, dtype=board.dtype) * -current_player, -1)
        return np.concatenate((side, np.expand_dims(board, -1)), axis=-1)

    def check_win(self):
        return self.check_win_MCTS(self.board, -self.next_player, None)

    @staticmethod
    def check_win_MCTS(board, current_player, action_history):
        """any complete line -> current_player (whoever owns it), full board -> 0, else -2 (Tictactoe.py:273-300)"""
        b = np.asarray(board)
        lines = [b[0], b[1], b[2], b[:, 0], b[:, 1], b[:, 2], np.diag(b), np.diag(np.fliplr(b))]
        for ln in lines:
            if ln[0] != 0 and ln[0] == ln[1] == ln[2]:
                return current_player
        if np.all(b != 0):
            return 0
        return -2


class Connect4:
    """6x7, actions = column index (Connect4/Connect4.py:218-445)."""

    def __init__(self):
        self.board = np.zeros((6, 7), dtype=np.int8)
        self.next_player = -1
        self.action_history = []
        self.policy_shape = (7,)

    def get_next_player(self):
        return self.next_player

    def input_action(self):
        while True:
            try:
                action = int(input("Action: "))
                if np.sum(abs(self.board[:, action])) < 6:
                    return action
                print("Illegal move")
            except Exception:
                print("Try again")

    def get_legal_actions(self):
        return self.get_legal_actions_MCTS(self.board, self.next_player, np.array(self.action_history))

    @staticmethod
    def get_legal_actions_MCTS(board, next_player, action_history):
        filled = np.abs(board).sum(axis=0)
        return np.nonzero(filled < 6)[0].astype(np.int8)

    @staticmethod
    def get_legal_actions_policy_MCTS(board, current_player, action_history, policy, normalize=True, shuffle=False):
        legal_actions = np.nonzero(np.abs(board).sum(axis=0) < 6)[0].astype(np.int8)
        legal_policy = policy[legal_actions]
        if normalize:
            legal_policy = legal_policy / _seq_sum(legal_policy)
        return legal_actions, legal_policy

    def do_action(self, action):
        row = 5 - int(np.sum(np.abs(self.board[:, action])))
        self.board[row][action] = self.next_player
        self.next_player *= -1
        self.action_history.append(action)

    @staticmethod
    def do_action_MCTS(board, action, next_player):
        row = 5 - int(np.sum(np.abs(board[:, action])))
        board[row][action] = next_player
        return board

    def get_input_state(self):
        return self.get_input_state_MCTS(self.board, -self.next_player, np.array(self.action_history, dtype=np.int8))

    @staticmethod
    def get_input_state_MCTS(board, current_player, action_history):
        """(6, 7, 4): plane 3 = board, planes 2 / 1 = one / two moves undone, plane 0 = current_player - and once
        four or more moves were played plane 0 is OVERWRITTEN by "three moves undone" (index -4 wraps to 0,
        Connect4.py:327-346)."""
        planes = np.zeros((4, 6, 7), dtype=np.int8)
        planes[0] = current_player
        planes[-1] = board
        undo = min(len(action_history) - 1, 3)
        prev = np.array(board, dtype=np.int8, copy=True)
        for i in range(-1, -undo - 1, -1):
            x = int(action_history[i])
            y = int(np.nonzero(prev[:, x])[0][0])   # top stone of the column
            prev[y][x] = 0
            planes[i - 1] = prev
        return np.transpose(planes, (1, 2, 0))

    def check_win(self):
        return self.check_win_MCTS(self.board, -self.next_player, np.array(self.action_history))

    @staticmethod
    def check_win_MCTS(board, current_player, action_history):
        """four in a row through the top stone of the last column -> current_player; full board -> 0; else -2
        (Connect4.py:351-411; its +-3 windows always contain the new stone, so this is a run-through-the-stone test)"""
        x = int(action_history[-1])
        y = int(np.nonzero(board[:, x] == current_player)[0][0])
        for dx, dy in ((1, 0), (0, 1), (1, -1), (1, 1)):
            run = 1
            for s in (1, -1):
                cx, cy = x + s * dx, y + s * dy
                while 0 <= cx <= 6 and 0 <= cy <= 5 and board[cy][cx] == current_player:
                    run += 1
                    cx += s * dx
                    cy += s * dy
            if run >= 4:
                return current_player
        if np.all(board != 0):
            return 0
        return -2

    def compute_policy_improvement(self, statistics):
        policy = np.zeros(7, dtype=np.float32)
        for action, prob in statistics:
            policy[action] = prob
        return policy

    @staticmethod
    def augment_sample(board, policy):
        """the reference's pair: np.fliplr on (T, 6, 7, 4) flips axis 1 - the ROWS - a reference quirk that is kept
        (Connect4.py:414-445); policies (T, 7) are mirrored left-right."""
        board, policy = np.asarray(board), np.asarray(policy)
        return np.stack((board, np.fliplr(board))), np.stack((policy, np.fliplr(policy)))


def eval_symmetries(name):
    """Board symmetries for symmetric network evaluation (Engine.set_eval_symmetry), built from the board geometry:
    the 8 dihedral maps in `_dihedral8`'s order for Gomoku and TicTacToe, the identity and the left-right column mirror
    of all four planes for Connect4 (not Connect4.augment_sample, whose np.fliplr flips the rows: an upside-down board is
    not a symmetry of the game).  Row 0 is the identity.  Returns (perm_state int32 (n, H*W*C), perm_policy int32 (n, P)):
        state_g[j] = state[perm_state[g][j]]    (the transformed HWC input state, flattened)
        p[a]       = q_g[perm_policy[g][a]]     (q_g = the network's policy row for state_g, p = the row mapped back)
    so perm_policy[g][a] is the action that a takes to under symmetry g."""
    H, W, C = {"gomoku": (15, 15, 2), "tictactoe": (3, 3, 2), "connect4": (6, 7, 4)}[name]
    cells = np.arange(H * W).reshape(H, W)
    maps = [cells, cells[:, ::-1]] if name == "connect4" else _dihedral8(cells)
    perm_state, perm_policy = [], []
    for m in maps:
        src = np.ascontiguousarray(m).reshape(-1)                # cell c of the transformed board = cell src[c]
        perm_state.append((src[:, None] * C + np.arange(C)).reshape(-1))
        inv = np.empty_like(src)
        inv[src] = np.arange(H * W)                              # original cell a sits at cell inv[a] of the transformed one
        perm_policy.append(inv if name != "connect4" else inv[:W])
    return np.array(perm_state, np.int32), np.array(perm_policy, np.int32)


GAME_NAMES = {Gomoku: "gomoku", Connect4: "connect4", TicTacToe: "tictactoe"}


def game_name_of(game):
    """engine game name of any object with the reference game interface (ours or the reference's own class)"""
    shape = tuple(np.shape(game.board))
    name = {(15, 15): "gomoku", (6, 7): "connect4", (3, 3): "tictactoe"}.get(shape)
    if name is None:
        raise ValueError("unsupported game: board shape %r (supported: Gomoku 15x15, Connect4 6x7, TicTacToe 3x3)" % (shape,))
    return name


def action_to_id(name, action):
    """reference action -> engine action id (cell index y*W+x, or the column)"""
    if name == "connect4":
        return int(action)
    w = 15 if name == "gomoku" else 3
    return int(action[1]) * w + int(action[0])


def id_to_action(name, a):
    """engine action id -> the reference's action object (Gomoku uint8 (x, y), TicTacToe int64 (x, y), Connect4 int8)"""
    if name == "connect4":
        return np.int8(a)
    if name == "gomoku":
        return np.array([a % 15, a // 15], dtype=np.uint8)
    return np.array([a % 3, a // 3], dtype=np.int64)
