"""Python twin of the symmetry choice of GAZ_SYM_RANDOM (TEST INFRASTRUCTURE ONLY).

Bit for bit the same function as ``sym_draw`` in grok_alpha_zero_b200/csrc/gaz_net.cu: the symmetry g under which a
request is evaluated is a hash of the seed of gaz_set_eval_symmetry, the tree's key (gaz_set_tree_keys, or seed ^ tree)
and the request's input-state bytes:
  acc = sum over the 8-byte little-endian words w_i of the int8 state (zero-padded) of mix(w_i + (i + 1) * GOLD) mod 2^64
  h   = mix(mix(mix(seed + GOLD) ^ key) ^ acc)
  g   = (h >> 32) % n
with mix the splitmix64 finaliser.
"""
import numpy as np

from hash_eval import GOLD, _M64, _mix_arr, _mix_int


def tree_key(seed, tree, tree_keys=None):
    """key of tree `tree`: tree_keys[tree] when the engine has per-tree keys, else seed ^ tree"""
    return int(tree_keys[tree]) if tree_keys is not None else (int(seed) ^ int(tree)) & _M64


def sym_draw(state, seed, key, n):
    """state: the request's input state (any int8-valued array, HWC); returns g in [0, n)"""
    b = np.asarray(state).astype(np.int8).reshape(-1).view(np.uint8)
    words = np.zeros((b.size + 7) // 8 * 8, np.uint8)
    words[:b.size] = b
    w = words.view("<u8").astype(np.uint64)
    with np.errstate(over="ignore"):
        terms = _mix_arr(w + (np.arange(1, w.size + 1, dtype=np.uint64) * np.uint64(GOLD)))
        acc = int(terms.sum(dtype=np.uint64))
    h = _mix_int(_mix_int(_mix_int((int(seed) + GOLD) & _M64) ^ (int(key) & _M64)) ^ acc)
    return int((h >> 32) % n)
