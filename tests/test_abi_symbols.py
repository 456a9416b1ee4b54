"""The C-ABI boundary: libgaz_b200.so loads on a GPU-less host and exports every function that include/*.h
declares; the ctypes tables (`_lib.SYMBOLS`, `_net_symbols.SYMBOLS`) name exactly those functions and agree with
the headers on the number of arguments.  No compute call is made (there is no GPU here and no CPU fallback:
`gaz_create` must fail loudly instead)."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from grok_alpha_zero_b200 import _lib, _net_symbols  # noqa: E402

HEADERS = {"gaz_b200.h": _lib.SYMBOLS, "gaz_net.h": _net_symbols.SYMBOLS}


def declared(header):
    """{function name: number of parameters} of the prototypes in include/<header>"""
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    out = {}
    for m in re.finditer(r"\b(gaz_\w+)\s*\(([^;{}]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
    return out


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()            # no-op when the library is newer than every source, rebuilds it otherwise
    return C.CDLL(ge.LIB)


@pytest.mark.parametrize("header", sorted(HEADERS))
def test_every_declared_symbol_is_exported(lib, header):
    names = declared(header)
    assert len(names) >= 10
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


@pytest.mark.parametrize("header", sorted(HEADERS))
def test_ctypes_tables_match_the_headers(header):
    names, table = declared(header), HEADERS[header]
    assert set(names) == set(table), (sorted(set(names) ^ set(table)))
    for n, nargs in names.items():
        assert len(table[n][1]) == nargs, (n, nargs, len(table[n][1]))


NO_DEVICE_CREATE = r'''
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from grok_alpha_zero_b200 import _lib
lib = C.CDLL(sys.argv[2])
cfg = _lib.GazConfig(game=0, mode=0, n_games=1, trees_per_game=1, node_cap=64, slot_cap=640, device=0, lut_n=64,
                     c_puct_init=2.5, c_puct_base=19652.0, gumbel_m=16, use_softmax=0, c_visit=50.0, c_scale=1.0)
h = C.c_void_p()
lib.gaz_create.restype = C.c_int
lib.gaz_create.argtypes = [C.POINTER(_lib.GazConfig), C.POINTER(C.c_void_p)]
rc = lib.gaz_create(C.byref(cfg), C.byref(h))
assert rc != 0 and not h.value                       # no device -> error code, never a CPU engine
lib.gaz_last_error.restype = C.c_char_p
assert lib.gaz_last_error()
'''


def test_abi_version_and_loud_failure_without_a_gpu(lib):
    lib.gaz_abi_version.restype = C.c_int
    assert lib.gaz_abi_version() >= 1
    # a child process with every device hidden: the same check runs on a GPU-less host and on a GPU machine
    import __graft_entry__ as ge
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_CREATE, ROOT, ge.LIB], env=env, capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
