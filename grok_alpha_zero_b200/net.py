"""Host side of the CUDA policy/value network: turns (netspec spec, Keras-layout weights) into the op
list + weight blobs of include/gaz_net.h and wraps the C ABI.

Replaces the evaluator behind the reference's session duck type
(MCTS.py:224-235 `session.run(["policy","value"], {"inputs": x})`), i.e. the onnxruntime session of
Self_Play.py:288-323 / Client_Server.py:119-120,206.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._net_symbols import GazNetBuf, GazNetDesc, GazNetOp
from .engine import GAMES, EngineError
from .netspec import bn_affine, is_tensor_core_conv, round_bf16

OP_STEM, OP_CONV_TC, OP_SE, OP_HEADCONV, OP_DENSE, OP_POLICY_OUT = range(6)
BUF_ROWS_BF16, BUF_ROWS_F32, BUF_FLAT_F32 = range(3)
ACT = {"none": 0, "relu": 1, "gelu": 2, "tanh": 3}
POLICY_MODE = {"softmax": 0, "stablemax": 1, "linear": 2}


def f32_to_bf16_bits(a):
    u = round_bf16(a).view(np.uint32)
    return (u >> 16).astype(np.uint16)


class _Builder:
    def __init__(self):
        self.wf = []
        self.n_wf = 0
        self.wh = []
        self.n_wh = 0
        self.bufs = []
        self.ops = []

    def f(self, arr):
        a = np.ascontiguousarray(arr, dtype=np.float32).reshape(-1)
        off = self.n_wf
        self.wf.append(a)
        self.n_wf += a.size
        pad = (-self.n_wf) % 4  # keep 16-byte alignment for vector loads
        if pad:
            self.wf.append(np.zeros(pad, np.float32))
            self.n_wf += pad
        return off

    def h(self, arr):
        a = f32_to_bf16_bits(np.ascontiguousarray(arr, dtype=np.float32)).reshape(-1)
        off = self.n_wh
        self.wh.append(a)
        self.n_wh += a.size
        pad = (-self.n_wh) % 64  # TMA global address alignment (128 B)
        if pad:
            self.wh.append(np.zeros(pad, np.uint16))
            self.n_wh += pad
        return off

    def buf(self, kind, width):
        self.bufs.append((kind, width))
        return len(self.bufs) - 1

    def op(self, type, **kw):
        d = dict(type=type, in_buf=-1, res_buf=-1, out_raw=-1, out_a=-1, out_b=-1, cin=0, cout=0, ksize=1, act=0,
                 flags=0, pad=0, w=-1, bias=-1, scale_a=-1, shift_a=-1, scale_b=-1, shift_b=-1, w2=-1, bias2=-1,
                 w3=-1, bias3=-1)
        d.update(kw)
        self.ops.append(d)


def build_ops(spec, W):
    """spec/weights -> (_Builder).  See include/gaz_net.h for the op semantics."""
    B = _Builder()
    layers = spec["layers"]
    stem = layers[0]
    blocks = [l for l in layers if l["op"] == "block"]
    heads = [l for l in layers if l["op"] == "head"]
    F = blocks[0]["cout"]
    SF = stem["cout"]

    def aff(name):
        s, t = bn_affine(W, name)
        return B.f(s), B.f(t)

    def tc_weights(name, k):
        kern = W[name + ".kernel"]  # (kh, kw, cin, cout) -> [cout][taps*cin]
        return B.h(np.transpose(kern, (3, 0, 1, 2)).reshape(kern.shape[3], -1))

    # which fused activations does the trunk's last block have to emit?
    head_pre = []  # (head, affine name) for heads that start with bnrelu + tensor-core conv
    for hd in heads:
        hl = hd["layers"]
        if hl[0]["t"] == "bnrelu" and hl[1]["t"] == "conv" and is_tensor_core_conv(hl[1]["cin"], hl[1]["cout"]):
            head_pre.append((hd["name"], hl[0]["name"]))
    assert len(head_pre) <= 2

    a_x = B.buf(BUF_ROWS_BF16, F)
    a_h = B.buf(BUF_ROWS_BF16, F)
    res = [B.buf(BUF_ROWS_F32, F), B.buf(BUF_ROWS_F32, F)]
    use_se = any(b["se"] for b in blocks)
    c2buf = B.buf(BUF_ROWS_F32, F) if use_se else -1
    head_in = {name: B.buf(BUF_ROWS_BF16, F) for name, _ in head_pre}

    # ---- stem
    first = blocks[0]
    sa, ta = aff(first["name"] + ".bn1")
    ss, ts = aff(stem["bn"])
    if first["proj"]:
        a_stem = B.buf(BUF_ROWS_BF16, SF)
        q_stem = B.buf(BUF_ROWS_BF16, SF)
        B.op(OP_STEM, cin=stem["cin"], cout=SF, ksize=stem["k"], act=ACT[stem["act"]], w=B.f(W[stem["name"] + ".kernel"]),
             bias=B.f(W[stem["name"] + ".bias"]), scale_b=ss, shift_b=ts, out_b=q_stem, out_a=a_stem, scale_a=sa, shift_a=ta)
        ain, rin = a_stem, -1
    else:
        B.op(OP_STEM, cin=stem["cin"], cout=SF, ksize=stem["k"], act=ACT[stem["act"]], w=B.f(W[stem["name"] + ".kernel"]),
             bias=B.f(W[stem["name"] + ".bias"]), scale_b=ss, shift_b=ts, out_raw=res[0], out_a=a_x, scale_a=sa, shift_a=ta)
        ain, rin = a_x, res[0]
        q_stem = -1
    # ---- blocks
    cur = 0 if rin == res[0] else -1
    for bi, b in enumerate(blocks):
        n = b["name"]
        if b["proj"]:
            tgt = res[0]
            B.op(OP_CONV_TC, in_buf=q_stem, out_raw=tgt, cin=b["cin"], cout=b["cout"], ksize=1,
                 w=tc_weights(n + ".proj", 1), bias=B.f(W[n + ".proj.bias"]))
            rin, cur = tgt, 0
        s2, t2 = aff(n + ".bn2")
        B.op(OP_CONV_TC, in_buf=ain, out_a=a_h, cin=b["cin"], cout=b["cout"], ksize=3, w=tc_weights(n + ".conv1", 3),
             bias=B.f(W[n + ".conv1.bias"]), scale_a=s2, shift_a=t2)
        rout = res[1 - cur]
        last = bi == len(blocks) - 1
        outs = {}
        if not last:
            sA, tA = aff(blocks[bi + 1]["name"] + ".bn1")
            outs = dict(out_a=a_x, scale_a=sA, shift_a=tA)
        else:
            for slot, (hname, bnname) in zip("ab", head_pre):
                sA, tA = aff(bnname)
                outs["out_" + slot] = head_in[hname]
                outs["scale_" + slot] = sA
                outs["shift_" + slot] = tA
        if b["se"]:
            B.op(OP_CONV_TC, in_buf=a_h, out_raw=c2buf, cin=b["cout"], cout=b["cout"], ksize=3,
                 w=tc_weights(n + ".conv2", 3), bias=B.f(W[n + ".conv2.bias"]))
            B.op(OP_SE, in_buf=c2buf, res_buf=rin, out_raw=rout, cin=b["cout"] // 2, cout=b["cout"],
                 w2=B.f(W[n + ".se1.kernel"]), bias2=B.f(W[n + ".se1.bias"]), w3=B.f(W[n + ".se2.kernel"]),
                 bias3=B.f(W[n + ".se2.bias"]), **outs)
        else:
            B.op(OP_CONV_TC, in_buf=a_h, res_buf=rin, out_raw=rout, cin=b["cout"], cout=b["cout"], ksize=3,
                 w=tc_weights(n + ".conv2", 3), bias=B.f(W[n + ".conv2.bias"]), **outs)
        ain, rin, cur = a_x, rout, 1 - cur
    x_raw = rin
    # ---- heads
    H, Wd = spec["H"], spec["W"]
    for hd in heads:
        hl = list(hd["layers"])
        i = 0
        cur_rows = x_raw        # padded-rows tensor the next conv reads
        if hd["name"] in head_in:  # bnrelu fused into the trunk epilogue, then a tensor-core conv
            conv = hl[1]
            nxt = hl[2]
            assert nxt["t"] == "bnrelu"
            sA, tA = aff(nxt["name"])
            mid = B.buf(BUF_ROWS_BF16, conv["cout"])
            B.op(OP_CONV_TC, in_buf=head_in[hd["name"]], out_a=mid, cin=conv["cin"], cout=conv["cout"], ksize=conv["k"],
                 w=tc_weights(conv["name"], conv["k"]), bias=B.f(W[conv["name"] + ".bias"]), scale_a=sA, shift_a=tA)
            cur_rows = mid
            i = 3
        conv = hl[i]
        assert conv["t"] == "conv", "head %s: expected a small conv at %d" % (hd["name"], i)
        kern = W[conv["name"] + ".kernel"].astype(np.float32)
        bias = W[conv["name"] + ".bias"].astype(np.float32)
        i += 1
        if hl[i]["t"] == "bn":  # channel BN right after the conv: fold (TicTacToe/Build_Model.py:33-34)
            s, t = bn_affine(W, hl[i]["name"])
            kern = kern * s[None, None, None, :]
            bias = bias * s + t
            i += 1
        assert hl[i]["t"] == "flatten"
        i += 1
        flat = B.buf(BUF_FLAT_F32, H * Wd * conv["cout"])
        B.op(OP_HEADCONV, in_buf=cur_rows, out_raw=flat, cin=conv["cin"], cout=conv["cout"], ksize=conv["k"],
             w=B.f(kern), bias=B.f(bias))
        pend_aff, pend_relu = None, False
        dense_layers = [l for l in hl[i:] if l["t"] == "dense"]
        cur_flat = flat
        for l in hl[i:]:
            if l["t"] == "bnrelu":
                pend_aff, pend_relu = l["name"], True
            elif l["t"] == "relu":
                pend_relu = True
            elif l["t"] == "dense":
                is_last = l is dense_layers[-1]
                kw = dict(in_buf=cur_flat, cin=l["cin"], cout=l["cout"], w=B.f(W[l["name"] + ".kernel"]),
                          bias=B.f(W[l["name"] + ".bias"]))
                flags = 0
                if pend_aff is not None:
                    s, t = aff(pend_aff)
                    kw.update(scale_a=s, shift_a=t)
                    flags |= 1
                if pend_relu:
                    flags |= 2
                if is_last and hd["out"] == "value":
                    flags |= 4
                    kw["act"] = ACT["tanh"]
                else:
                    nb = B.buf(BUF_FLAT_F32, l["cout"])
                    kw["out_raw"] = nb
                    cur_flat = nb
                B.op(OP_DENSE, flags=flags, **kw)
                pend_aff, pend_relu = None, False
        if hd["out"] == "policy":
            B.op(OP_POLICY_OUT, in_buf=cur_flat)
    return B


def check_weights(spec, W):
    """Every array the network reads must be present with the shape `spec` implies: a dictionary built for another
    build_config would otherwise be re-laid-out into operands of the wrong size."""
    from .keras_bridge import expected_shapes
    want = expected_shapes(spec)
    for l in spec["layers"]:
        if l["op"] == "block" and l["se"]:
            r = l["cout"] // 2
            want.update({l["name"] + ".se1.kernel": (l["cout"], r), l["name"] + ".se1.bias": (r,),
                         l["name"] + ".se2.kernel": (r, l["cout"]), l["name"] + ".se2.bias": (l["cout"],)})
    for k, shp in want.items():
        if k not in W:
            raise ValueError("network weights: %r is missing (spec %s %s)" % (k, spec["game"], spec["cfg"]))
        if tuple(np.shape(W[k])) != tuple(shp):
            raise ValueError("network weights: %r has shape %s, the spec (%s %s) expects %s"
                             % (k, tuple(np.shape(W[k])), spec["game"], spec["cfg"], tuple(shp)))


class Net:
    """CUDA policy/value network.  `forward` is the host-buffer path (parity tests, mailbox server);
    `attach(engine)` wires it to a search engine so leaves never leave HBM.

    `share=net` uses `net`'s activation workspace (everything that scales with `max_batch`) instead of allocating one: the
    spec must be structurally the same (same game, layers and widths; the weights may differ), with the same `max_batch`
    and device.  The workspace lives until the last network using it is closed.  Networks sharing a workspace must not run
    forward passes at the same time; networks attached to one engine never do, and `forward` returns synchronised."""

    def __init__(self, spec, weights, max_batch, device=0, lib=None, share=None):
        self.lib = lib if lib is not None else _lib.load()
        self.spec = spec
        self.H, self.W, self.Cin, self.P = spec["H"], spec["W"], spec["Cin"], spec["P"]
        self.max_batch = max_batch
        check_weights(spec, weights)
        b = build_ops(spec, weights)
        self.n_ops = len(b.ops)
        self.n_conv_tc = sum(1 for o in b.ops if o["type"] == OP_CONV_TC)
        self.conv_shapes = [(o["cin"], o["cout"], o["ksize"]) for o in b.ops if o["type"] == OP_CONV_TC]
        # (type, cin, cout, ksize, tag): tag "se" = convolution whose epilogue carries the following SE op; "block" = conv1
        # that runs the whole residual block (conv1 + conv2 + SE + skip, gaz_block.cuh) and "inblock" = the conv2 it absorbed.
        # Mirrors the fusion rules of gaz_net_create (csrc/gaz_net.cu).
        p_pad = (spec["H"] + 1) * (spec["W"] + 1)       # rows per board, rounded up to a divisor of the 256-row tile (gaz_net_create)
        if p_pad <= 256:
            r = 16
            while r < p_pad:
                r <<= 1
            p_pad = r
        tile_is_board = p_pad == 256
        fuse_block = 256 % p_pad == 0
        self._op_shapes = []
        for i, o in enumerate(b.ops):
            tag = ""
            if o["type"] == OP_CONV_TC and i + 1 < len(b.ops) and b.ops[i + 1]["type"] == OP_SE and tile_is_board:
                tag = "se"
            self._op_shapes.append([o["type"], o["cin"], o["cout"], o["ksize"], tag])
        if fuse_block:
            for i in range(len(b.ops) - 1):
                o, o2 = b.ops[i], b.ops[i + 1]
                if o["type"] == OP_CONV_TC and o2["type"] == OP_CONV_TC and (o["cin"], o["cout"], o["ksize"]) in ((128, 128, 3), (256, 128, 3)) and \
                        (o2["cin"], o2["cout"], o2["ksize"]) == (128, 128, 3) and o["out_a"] >= 0 and o["out_b"] < 0 and \
                        o["out_raw"] < 0 and o["res_buf"] < 0 and o2["in_buf"] == o["out_a"] and self._op_shapes[i][4] == "":
                    self._op_shapes[i][4] = "block+" + self._op_shapes[i + 1][4]
                    self._op_shapes[i + 1][4] = "inblock"
        self._op_shapes = [tuple(x) for x in self._op_shapes]
        bufs = (GazNetBuf * len(b.bufs))(*[GazNetBuf(k, w) for k, w in b.bufs])
        ops = (GazNetOp * len(b.ops))(*[GazNetOp(**o) for o in b.ops])
        wf = np.concatenate(b.wf) if b.wf else np.zeros(4, np.float32)
        wh = np.concatenate(b.wh) if b.wh else np.zeros(64, np.uint16)
        desc = GazNetDesc(GAMES[spec["game"]], max_batch, len(b.bufs), len(b.ops), POLICY_MODE[spec["policy_head"]],
                          device, bufs, ops, wf.ctypes.data_as(C.c_void_p), wf.size, wh.ctypes.data_as(C.c_void_p),
                          wh.size)
        h = C.c_void_p()
        self._h = None
        if share is not None and share._h is None:
            raise ValueError("share: that network is closed")
        rc = self.lib.gaz_net_create_shared(C.byref(desc), share._h if share is not None else None, C.byref(h))
        if rc < 0:
            raise EngineError(self.lib.gaz_last_error().decode())
        self._h = h
        self.n_launches = int(self.lib.gaz_net_launches_per_forward(h))   # kernels per forward (fused ops launch nothing)
        # consecutive fused blocks share a launch (trunk launches, gaz_block.cuh): "block+se*5" = this op's launch runs 5 blocks,
        # "intrunk" = the block runs inside an earlier op's launch
        shapes = [list(x) for x in self._op_shapes]
        for i, x in enumerate(shapes):
            if x[4].startswith("block"):
                nb = int(self.lib.gaz_net_op_blocks(h, i))
                x[4] = "intrunk" if nb == 0 else (x[4] + "*%d" % nb)
        self._op_shapes = [tuple(x) for x in shapes]

    def _ck(self, rc):
        if rc < 0:
            raise EngineError(self.lib.gaz_last_error().decode())
        return rc

    def close(self):
        if self._h is not None:
            self.lib.gaz_net_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def forward(self, states, want_logits=False):
        st = np.ascontiguousarray(states, dtype=np.int8).reshape(-1, self.H, self.W, self.Cin)
        n = st.shape[0]
        pol = np.zeros((n, self.P), np.float32)
        val = np.zeros(n, np.float32)
        lg = np.zeros((n, self.P), np.float32) if want_logits else None
        self._ck(self.lib.gaz_net_forward_host(self._h, st.ctypes.data_as(C.c_void_p), n,
                                               pol.ctypes.data_as(C.c_void_p), val.ctypes.data_as(C.c_void_p),
                                               lg.ctypes.data_as(C.c_void_p) if want_logits else None))
        return (pol, val, lg) if want_logits else (pol, val)

    def attach(self, engine):
        self._ck(self.lib.gaz_attach_net(engine._h, self._h))
        engine._net = self  # keep alive

    def op_shapes(self):
        """(op type, cin, cout, ksize, tag) of every op in launch order"""
        return list(self._op_shapes)

    def bytes_allocated(self):
        return int(self.lib.gaz_net_bytes(self._h))

    def profile(self, max_launches):
        self._ck(self.lib.gaz_net_profile(self._h, int(max_launches)))

    def profile_read(self):
        tot = C.c_float()
        cnt = C.c_int()
        per = np.zeros(self.n_ops, np.float32)
        self._ck(self.lib.gaz_net_profile_read(self._h, C.byref(tot), C.byref(cnt), per.ctypes.data_as(C.c_void_p)))
        return float(tot.value), int(cnt.value), per

    def time_forward(self, n, iters=10):
        ms = np.zeros(2, np.float32)
        self._ck(self.lib.gaz_net_time_forward(self._h, int(n), int(iters), ms.ctypes.data_as(C.c_void_p)))
        return float(ms[0])
