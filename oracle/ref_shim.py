"""Import the UNMODIFIED reference from /root/reference (TEST INFRASTRUCTURE ONLY).

Works only in the build container (the GPU box has no /root/reference); used by
oracle/gen_golden.py, gen_cache_golden.py and gen_selfplay_golden.py to produce fixtures under tests/golden/.
Recipe: SURVEY.md section 8(c).
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("GAZ_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isdir(REFERENCE_ROOT) and os.path.exists(os.path.join(REFERENCE_ROOT, "MCTS.py"))


def load():
    """Returns a namespace with MCTS, MCTS_Gumbel and the three game classes."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/ref_nbcache")  # reference dir is read-only
    if "onnxruntime" not in sys.modules:
        ort = types.ModuleType("onnxruntime")
        ort.InferenceSession = type("InferenceSession", (), {})
        sys.modules["onnxruntime"] = ort  # only used for annotations at import (MCTS.py:16)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import numpy as np
    from MCTS import MCTS
    from MCTS_Gumbel import MCTS_Gumbel
    from Gomoku.Gomoku import Gomoku
    from Connect4.Connect4 import Connect4
    from TicTacToe.Tictactoe import TicTacToe

    # parity rule: lowest-index terminal child (MCTS.py:208).  np.random.randint is
    # swapped only while _PUCT_select runs (numba's own np.random typing needs the real one).
    orig_select = MCTS._PUCT_select

    def _select_lowest_terminal(self):
        saved = np.random.randint
        np.random.randint = lambda low=0, high=None, **k: low
        try:
            return orig_select(self)
        finally:
            np.random.randint = saved

    MCTS._PUCT_select = _select_lowest_terminal
    ns = types.SimpleNamespace(MCTS=MCTS, MCTS_Gumbel=MCTS_Gumbel, Gomoku=Gomoku, Connect4=Connect4,
                               TicTacToe=TicTacToe)
    ns.games = {"tictactoe": TicTacToe, "connect4": Connect4, "gomoku": Gomoku}
    return ns
