#!/usr/bin/env python
"""bench.py -- MCTS simulations/s of the self-play hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config gomoku|connect4|gumbel|tictactoe] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # CPU arm: the oracle port of the reference path on the host cores

Workload (BASELINE.json configs[2], the config the north-star target is quoted on): Gomoku 15x15 self-play,
PUCT with 800 sims/move (Self_Play.py:99 passes int(800*1.5) = 1200 iterations), 10-block ResNet(128)+SE in
bf16, 16384 concurrent games per GPU, two trees per game as in Self_Play.py:39-57, random-init synthetic
weights (no checkpoint exists anywhere).  Games shard over GPUs by index with no collective on the search
path (SURVEY 8e), so scaling is "weak": per-GPU work is fixed.

A STEP is one search round: one simulation in every running tree = select (PUCT descent, terminal
look-ahead, leaf encode) -> network forward on the gathered leaves -> expand + backup.  `value` counts the
simulations the device actually performed (iteration counters read back), divided by the CUDA-event time of
the K timed rounds on the engine's stream, max over ranks.  When a run reaches its iteration limit inside the
timed region the move transition (root stats -> argmax move -> apply -> re-root both trees -> next run)
happens inside the timed region too.

`e2e` is the same metric through the public host-buffer API: every e2e pass uploads all live game boards from
pinned host memory (gaz_set_games), builds fresh roots (1 evaluation each, the MCTS constructor of
MCTS.py:132), runs K rounds and reads every root's visit counts / value sums / chosen move back to the host
(gaz_root_dense).  Root construction and both copies are inside its timed region; only the K*games
simulations are counted.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: game, mode, games/GPU, sims/move, iteration limit handed to run(), net overrides, c_puct, opening
    "gomoku": dict(game="gomoku", mode="puct", games=16384, sims=800, limit=1200, net={}, head="softmax",
                   c_puct_init=4.5, alpha=0.05, opening=112, label="Gomoku 15x15 self-play, PUCT 800 sims/move (x1.5 = 1200 "
                   "iterations, Self_Play.py:99), 10-block ResNet128+SE bf16, 16384 games/GPU"),
    # the reference's own Gomoku builder has no Squeeze-Excitation (Gomoku/Build_Model.py:10-88): same trunk without the SE epilogue
    "gomoku_no_se": dict(game="gomoku", mode="puct", games=16384, sims=800, limit=1200, net=dict(use_se=False), head="softmax",
                         c_puct_init=4.5, alpha=0.05, opening=112, label="Gomoku 15x15 self-play, PUCT 800 sims/move (x1.5 = 1200 "
                         "iterations), 10-block ResNet128 WITHOUT SE (the reference's builder) bf16, 16384 games/GPU"),
    "connect4": dict(game="connect4", mode="puct", games=4096, sims=800, limit=1200, net={}, head="softmax",
                     c_puct_init=2.5, alpha=0.5, opening=None, label="Connect4 6x7 self-play, PUCT 800 sims/move, 5-block "
                     "ResNet128 bf16, 4096 games/GPU"),
    "gumbel": dict(game="gomoku", mode="gumbel", games=16384, sims=64, limit=64, net={}, head="stablemax",
                   c_puct_init=4.5, alpha=None, opening=112, label="Gomoku 15x15 Gumbel MCTS m=16 n=64 StableMax, 10-block "
                   "ResNet128+SE bf16, 16384 games/GPU"),
    "tictactoe": dict(game="tictactoe", mode="puct", games=4096, sims=200, limit=300, net={}, head="softmax",
                      c_puct_init=1.25, alpha=1.0, opening=None, label="TicTacToe 3x3 self-play, PUCT 200 sims/move, small "
                      "ResNet, 4096 games/GPU"),
}


def kernel_sha16():
    """hash of the tcgen05 kernel sources: ties profiles/conv_traffic.json (an ncu capture) to the code it was taken on"""
    import hashlib
    h = hashlib.sha256()
    for f in ("gaz_tc.cuh", "gaz_conv.cuh", "gaz_block.cuh"):
        h.update(open(os.path.join(ROOT, "grok_alpha_zero_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, burst=1590.0, sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)),
                    samples=len(sm), reasons=sorted(reasons))


def tree_caps(cfg):
    """(node_cap, slot_cap) per tree: the rule of Self_Play.BatchedSelfPlay, i.e. pools sized for the tail of WHOLE games
    (measured peaks at 1200 iterations/move: 2806 nodes / 374 k child slots in 12 emulated Gomoku games), not for the
    opening the timed region happens to lie in - the HBM footprint in `hbm_bytes` is what a real generation needs."""
    lim = cfg["limit"]
    if cfg["game"] == "gomoku":
        if cfg["mode"] == "gumbel":
            n = int(lim * 1.5) + 2 * 225 + 64
            return n, n * 225 + 256
        return 4 * lim + 4 * 225 + 64, 2 * lim * 225 + 256
    L = 7 if cfg["game"] == "connect4" else 9
    n = 8 * lim + 4 * L + 64
    return n, n * L + 256


class SelfPlayBench:
    """Drives the engine the way Self_Play.play does (two PUCT trees per game, the tree of the side to move
    searches, both are re-rooted after the move; one fresh Gumbel tree per move)."""

    def __init__(self, cfg, n_games, device, noise=True, pool_fraction=1.0, eval_cache=0, keep_roots=False):
        from grok_alpha_zero_b200 import netspec
        from grok_alpha_zero_b200.engine import Engine
        from grok_alpha_zero_b200.net import Net
        self.cfg, self.n_games = cfg, n_games
        self.gumbel = cfg["mode"] == "gumbel"
        self.tpg = 1 if self.gumbel else 2
        self.spec = netspec.build_spec(cfg["game"], cfg["head"] if not self.gumbel else "linear", **cfg["net"])
        self.weights = netspec.init_weights(self.spec, seed=0)
        self.flops_per_eval = netspec.flops_per_eval(self.spec)
        node_cap, slot_cap = tree_caps(cfg)
        # child slots live in an engine-wide page pool (include/gaz_b200.h gaz_config.slot_pool); fraction 1.0 = every tree can
        # reach its per-tree limit at once, < 1 sizes the pool from the mean occupancy (more games per GPU)
        slot_pool = 0 if pool_fraction >= 1.0 else int(pool_fraction * n_games * self.tpg * slot_cap)
        self.eng = Engine(cfg["game"], n_games=n_games, mode=cfg["mode"], trees_per_game=self.tpg, node_cap=node_cap,
                          slot_cap=slot_cap, c_puct_init=cfg["c_puct_init"], m=16, c_visit=50.0, c_scale=1.0,
                          activation_fn="stablemax" if self.gumbel else "softmax", device=device, slot_pool=slot_pool)
        if eval_cache > 0:   # parity-safe evaluation dedup (per-game scope): OFF for the headline, reported separately
            self.eng.enable_eval_cache(eval_cache, shared=False)
        self.net = Net(self.spec, self.weights, max_batch=n_games, device=device)
        self.net.attach(self.eng)
        # exploration noise as Self_Play.py:38-69 configures the searches: Dirichlet(alpha) at every PUCT expansion
        # (device Philox streams keyed by the global game id), Gumbel(0,1) on the root logits of every Gumbel run
        self.noise = noise
        rank = int(os.environ.get("RANK", "0"))
        self.gumbel_noise = None
        if noise and not self.gumbel:
            gid = np.arange(n_games, dtype=np.uint64) + np.uint64(rank * n_games)
            self.eng.set_tree_keys(np.repeat(gid, self.tpg) * np.uint64(self.tpg) + np.tile(np.arange(self.tpg, dtype=np.uint64), n_games))
            self.eng.set_noise(cfg["alpha"], 0.25, seed=2024)
        if noise and self.gumbel:
            self.gumbel_noise = np.random.default_rng(2024 + rank).gumbel(size=(n_games, 256))
        self.moves = 0
        self.sims_done = 0       # simulations of finished runs
        self.next_player = np.full(n_games, -1, np.int32)
        self.alive = np.ones(n_games, bool)
        self.launches = 0
        # keep_roots: advance_move keeps the root statistics of the search it finishes (value sums included) in last_roots,
        # so that what a search handed its caller can still be read after the trees were re-rooted
        self.keep_roots, self.last_roots = keep_roots, None
        self.per_round_launches = 3 + 1 + self.net.n_launches  # counter reset, select, expand + chunk count + network kernels
        if eval_cache > 0:
            self.per_round_launches += 2                       # cache look-up and fill passes

    # ---- Self_Play.play pieces -------------------------------------------------------------
    def start(self):
        e, cfg = self.eng, self.cfg
        e.reset_games()
        if cfg["opening"] is not None:  # Gomoku/Gomoku.py:47 opening book [[7,7], 0.333]: every third game
            a = np.full(self.n_games, -1, np.int16)
            a[::3] = cfg["opening"]
            e.apply_actions(a)
            self.next_player[::3] = 1
        self._fresh_roots()
        self._begin_run()

    def _fresh_roots(self, mask=None):
        e = self.eng
        for k in range(self.tpg):  # one tree per game at a time keeps the batch <= n_games
            m = np.zeros((self.n_games, self.tpg), np.uint8)
            m[:, k] = 1 if mask is None else mask
            if e.new_roots(m.reshape(-1)) > 0:
                e.eval_net()
                self.launches += 1 + self.net.n_launches
            e.expand()
            self.launches += 3

    def _limits(self):
        lim = np.zeros((self.n_games, self.tpg), np.int32)
        if self.gumbel:
            lim[:, 0] = np.where(self.alive, self.cfg["limit"], 0)
        else:
            lim[np.arange(self.n_games), (self.next_player > 0).astype(int)] = np.where(self.alive, self.cfg["limit"], 0)
        return lim.reshape(-1)

    def _begin_run(self):
        if self.gumbel_noise is not None:   # MCTS_Gumbel.py:592-594; a fresh draw per move (rows rotate through one table)
            self.gumbel_noise = np.roll(self.gumbel_noise, 1, axis=0)
            self.eng.set_gumbel_noise(self.gumbel_noise)
        self.eng.run_begin(self._limits())
        self.launches += 1

    def rounds(self, n, sync=False):
        self.eng.rounds_net(n, sync=sync)
        self.launches += n * self.per_round_launches
        self.last_roots = None

    def run_finished(self):
        return self.eng.remaining() == 0

    def advance_move(self):
        """root stats -> tau=0 move -> do_action/check_win -> prune_tree on both trees -> next run"""
        e = self.eng
        vis, val, info = e.root_dense(want_values=self.keep_roots)
        if self.keep_roots:
            self.last_roots = (vis, val, info)
        info = info.reshape(self.n_games, self.tpg, 4)
        run_tree = 0 if self.gumbel else (self.next_player > 0).astype(int)
        sel = info[np.arange(self.n_games), run_tree]
        self.sims_done += int(sel[self.alive, 2].sum())
        act = np.where(self.alive, sel[:, 1], -1).astype(np.int16)
        winners = e.apply_actions(act)
        self.next_player = np.where(self.alive, -self.next_player, self.next_player)
        self.alive &= winners == -2
        self.moves += int((act >= 0).sum())
        pa = np.repeat(np.where(self.alive, act, -1).astype(np.int16), self.tpg)
        if e.prune(pa, create_new_root=self.gumbel) > 0:  # Gumbel: tree rebuilt every move (Self_Play.py:151-153)
            e.eval_net()
            self.launches += 1 + self.net.n_launches
        e.expand()
        self.launches += 6
        self._begin_run()

    def sims_in_flight(self):
        _, _, info = self.eng.root_dense(want_values=False)
        info = info.reshape(self.n_games, self.tpg, 4)
        run_tree = 0 if self.gumbel else (self.next_player > 0).astype(int)
        sel = info[np.arange(self.n_games), run_tree]
        return int(sel[self.alive, 2].sum())

    def evals_total(self):
        """evaluations the NETWORK performed: leaf requests minus the evaluation-cache hits"""
        _, _, info = self.eng.root_dense(want_values=False)
        return int(info[:, 3].astype(np.int64).sum()) - self.eng.eval_cache_stats()["hits"]

    def total_sims(self):
        return self.sims_done + self.sims_in_flight()


DUMP_LIMIT_BYTES = 64 * 10 ** 6 - 4096     # 64 MB less room for the .npy headers


def dump_outputs(sb, folder):
    """Root statistics of every tree after the last timed search round (gaz_root_dense: visit counts and value sums by action
    id, per-tree root visits / tau=0 move / iterations / evaluations), written as float32 / float64 .npy files so that two
    builds can be compared output for output.  If the timed region ended with a move transition, they are the statistics
    that move was chosen from, not those of the re-rooted trees.  Above 64 MB a fixed seeded sample of trees is written,
    with its tree indices."""
    vis, val, info = sb.last_roots if sb.last_roots is not None else sb.eng.root_dense(want_values=True)
    out = dict(root_visits=vis.astype(np.float32), root_value_sums=val.astype(np.float32), root_info=info.astype(np.float64))
    n_trees = vis.shape[0]
    row_bytes = sum(a[0].nbytes for a in out.values())
    keep = min(n_trees, (DUMP_LIMIT_BYTES - 8 * n_trees) // row_bytes)
    if keep < n_trees:
        rows = np.sort(np.random.default_rng(0).choice(n_trees, keep, replace=False))
        out = {k: a[rows] for k, a in out.items()}
        out["tree_index"] = rows.astype(np.float64)
    os.makedirs(folder, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(folder, k + ".npy"), a)


def dominant_kernel_stats(sb, leaves_per_launch, peaks):
    """CUDA-event time of the dominant kernel group inside the timed region.  Groups = tensor-core convolutions of
    one shape; the 3x3 C128->C128 launches are split into plain ones (block conv1) and those whose epilogue carries
    the Squeeze-Excitation + skip add (block conv2)."""
    tot, cnt, per = sb.net.profile_read()
    shapes = sb.net.op_shapes()
    groups = {}
    for oi, (typ, cin, cout, k, tag) in enumerate(shapes):
        if typ != 1 or per[oi] <= 0:
            continue
        g = groups.setdefault((cin, cout, k, tag), [0.0, 0])
        g[0] += float(per[oi])
        g[1] += 1
    if not groups:
        return None, {}
    n_tc_ops = sum(g[1] for g in groups.values())
    passes = cnt / max(1, n_tc_ops)
    hw = sb.spec["H"] * sb.spec["W"]

    def n_blocks(tag):      # "block+se*5": one launch runs 5 consecutive residual blocks (trunk launch, gaz_block.cuh)
        return int(tag.split("*")[1]) if "*" in tag else 1

    def label(cin, cout, k, tag):
        if tag.startswith("block"):
            nb = n_blocks(tag)
            tail = "+SE+skip" if "se" in tag else "+skip"
            if cin != cout:
                first = "residual block 3x3 C%d->C%d, 3x3 C%d->C%d%s" % (cin, cout, cout, cout, tail)
                return first if nb == 1 else "%s followed by %d x residual block 2x(3x3 C%d->C%d)%s, one launch" % (first, nb - 1, cout, cout, tail)
            return "%sresidual block 2x(3x3 C%d->C%d)%s" % ("%d x " % nb if nb > 1 else "", cin, cout, tail + (", one launch" if nb > 1 else ""))
        return "%dx%d C%d->C%d%s" % (k, k, cin, cout, "+SE" if tag == "se" else "")

    def work(cin, cout, k, tag):
        """algorithmic (FLOPs, HBM bytes over live cells) of one launch"""
        cells = leaves_per_launch * hw
        conv = 2.0 * cells * k * k * cin * cout
        if tag.startswith("block"):   # per block two convolutions; in: bf16 operand + fp32 residual, out: fp32 residual + bf16 operand
            nb = n_blocks(tag)
            inner = 2.0 * cells * k * k * cout * cout
            return (conv + inner) + (nb - 1) * 2.0 * inner, cells * ((cin * 2 + cout * 4 + cout * 4 + cout * 2) + (nb - 1) * (cout * 2 + cout * 4 + cout * 4 + cout * 2))
        if tag == "se":
            return conv, cells * (cin * 2 + cout * 4 + cout * 4 + cout * 2)
        return conv, cells * (cin * 2 + cout * 2)

    detail = {}
    for (cin, cout, k, tag), (ms, nops) in groups.items():
        launches = nops * passes
        avg_ms = ms / max(1.0, launches)
        fl, _ = work(cin, cout, k, tag)
        detail[label(cin, cout, k, tag)] = dict(launches=int(launches), avg_launch_ms=round(avg_ms, 4),
                                                tflops=round(fl / (avg_ms * 1e-3) / 1e12, 1),
                                                share_of_conv_time=round(ms / max(tot, 1e-9), 4))
    key = max(groups, key=lambda g: groups[g][0])
    cin, cout, k, tag = key
    launches = groups[key][1] * passes
    avg_ms = groups[key][0] / max(1.0, launches)
    flops, bytes_alg = work(cin, cout, k, tag)
    # DRAM bytes per launch come from an `ncu --set full` capture (bench.py cannot read DRAM counters itself); the record is
    # used only if it was taken on THESE kernel sources (hash of the tcgen05 headers) at this batch size, else null
    traffic = None
    tp = os.path.join(ROOT, "profiles", "conv_traffic.json")
    if os.path.exists(tp):
        try:
            tkey = "block_3x3_C%d_C%d_x%d" % (cin, cout, n_blocks(tag)) if tag.startswith("block") else "%dx%d_C%d_C%d%s" % (k, k, cin, cout, "_se" if tag else "")
            t = json.load(open(tp)).get(tkey)
            if t and t.get("leaves") == int(round(leaves_per_launch)) and t.get("kernel_sha16") == kernel_sha16():
                traffic = t.get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    if tag.startswith("block"):
        name = ("gaz_block::res_trunk_kernel, %d residual block(s) per launch (per block: conv1 -> SMEM -> conv2 + SE + skip, tcgen05 "
                "cta_group::2 implicit GEMMs)" % n_blocks(tag))
    else:
        name = ("gaz_conv::conv_board_kernel<%d, pair> %dx%d C%d->C%d%s (tcgen05 cta_group::2 implicit GEMM)"
                % (cout, k, k, cin, cout, " + fused SE/skip epilogue" if tag else ""))
    common = dict(kernel=name, avg_launch_ms=round(avg_ms, 4), launches_timed=int(launches),
                  share_of_conv_time=round(groups[key][0] / max(tot, 1e-9), 4), traffic=traffic, groups=detail)
    # the bound follows the arithmetic intensity: machine balance = sustained bf16 peak / HBM copy bandwidth
    balance = peaks["sustained"] * 1e12 / (peaks["hbm"] * 1e9)
    if flops / bytes_alg < balance:
        achieved = bytes_alg / (avg_ms * 1e-3) / 1e9
        roof = dict(bound="hbm", achieved=round(achieved, 1), peak=peaks["hbm"], unit="GB/s", frac=round(achieved / peaks["hbm"], 4),
                    peak_source="%s HBM copy bandwidth" % peaks["source"], bytes_per_launch=bytes_alg,
                    intensity_flop_per_byte=round(flops / bytes_alg, 1), machine_balance=round(balance, 1),
                    tensor_view=dict(tflops=round(flops / (avg_ms * 1e-3) / 1e12, 1), flops_per_launch=flops), **common)
    else:
        achieved = flops / (avg_ms * 1e-3) / 1e12
        roof = dict(bound="tensor", achieved=round(achieved, 2), peak=peaks["sustained"], unit="TFLOP/s",
                    frac=round(achieved / peaks["sustained"], 4),
                    peak_source="%s bf16 sustained (kernel timed inside a long step)" % peaks["source"],
                    flops_per_launch=flops, bytes_per_launch=bytes_alg, intensity_flop_per_byte=round(flops / bytes_alg, 1),
                    machine_balance=round(balance, 1), **common)
    return roof, dict(conv_ms_total=tot, conv_launches=cnt)


def run_reference(args, cfg):
    """CPU arm: oracle port of the reference path (numba MCTS + inference server) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import __graft_entry__ as ge
    ge.build_oracle()
    import cpu_selfplay
    from grok_alpha_zero_b200 import netspec
    cores = os.cpu_count() or 1
    workers = cores
    spec = netspec.build_spec(cfg["game"], cfg["head"], **cfg["net"])
    W = netspec.init_weights(spec, seed=0)
    sims_per_step = 4
    r = cpu_selfplay.run_sample(cfg["game"], spec, W, n_workers=workers, sims_per_step=sims_per_step, steps=args.steps,
                                warmup=args.warmup, c_puct_init=cfg["c_puct_init"], opening=cfg["opening"],
                                torch_threads=cores)
    sample = ("%d worker threads x 1 game (C oracle port of MCTS.py) + 1 batching inference server (fp32 torch-CPU "
              "restatement of the Keras net standing in for onnxruntime-CPU, mean batch %.1f); step = %d sims/game"
              % (workers, r["mean_batch"], sims_per_step))
    line = dict(impl="reference", metric="MCTS simulations/sec", value=r["sims_per_s"], unit="sims/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=r["ms_per_step"], higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=cfg["label"], reference_sample=sample),
                cpu_baseline=dict(value=r["sims_per_s"], unit="sims/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=r["sims_per_s"], unit="sims/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line), flush=True)


def run_moves(args, cfg, sb, timed_moves, barrier, world, rank, local, n_games):
    """--moves M: the timed region is M whole moves of every game (the first move is warm-up)."""
    import torch
    import torch.distributed as dist
    timed_moves(1)
    sims0, evals0, l0, m0 = sb.sims_done, sb.evals_total(), sb.launches, sb.moves
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    ms, rounds = timed_moves(args.moves)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    status = sb.eng.status()
    if status != 0:
        raise SystemExit("engine status %d (1 node overflow, 2 slot overflow, 4 LUT miss, 8 bad state)" % status)
    tot = torch.tensor([float(sb.sims_done - sims0), float(sb.evals_total() - evals0), float(sb.moves - m0),
                        float(sb.alive.sum())], dtype=torch.float64, device="cuda")
    mst = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(mst, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    line = None
    if rank == 0:
        sims, evals, moves, alive = (float(x) for x in tot.tolist())
        t = float(mst.item()) * 1e-3
        line = (dict(
            metric="MCTS simulations/sec", value=sims / t, unit="sims/s", n_gpus=world, steps=rounds, warmup=cfg["limit"],
            ms_per_step=t * 1e3 / rounds, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
            data="synthetic",
            config=dict(workload=cfg["label"], games_per_gpu=n_games, trees_per_game=sb.tpg,
                        step="one search round; timed region = %d whole moves of every game after one warm-up move "
                             "(search, move choice at tau=0, do_action/check_win, prune_tree of both trees, next run)" % args.moves,
                        noise="on" if sb.noise else "off"),
            positions_per_s=moves / t, moves_timed=int(moves), games_still_running=int(alive),
            nn_evals_per_s=evals / t, sims_per_eval=sims / max(1.0, evals), gpu_launches=int(sb.launches - l0),
            clocks=clocks, hbm_bytes=dict(engine=sb.eng.bytes_allocated(), net=sb.net.bytes_allocated()),
            eval_cache=(dict(sb.eng.eval_cache_stats(), scope="per game") if args.eval_cache > 0 else None)))
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed search rounds (default 40)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="gomoku", choices=sorted(CONFIGS))
    ap.add_argument("--games", type=int, default=0, help="override games per GPU")
    ap.add_argument("--presearch", type=int, default=-1,
                    help="untimed rounds before warm-up so trees are mid-search (default: past the forced root expansion)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--moves", type=int, default=0,
                    help="time M WHOLE moves per game from the start position (search, move choice, do_action, prune_tree / "
                         "re-rooting of both trees) instead of K rounds: positions/s measured directly; replaces --steps")
    ap.add_argument("--no-noise", action="store_true", help="searches without Dirichlet / Gumbel exploration noise")
    ap.add_argument("--eval-cache", type=int, default=0,
                    help="entries of the device-side evaluation cache (per-game scope; 0 = off, the default and the headline)")
    ap.add_argument("--pool-fraction", type=float, default=1.0,
                    help="size of the engine-wide child-slot page pool as a fraction of n_trees * slot_cap (1.0 = static worst case)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the sub-records of the default run (the other BASELINE configurations at N=1, the real generation at N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed region, write rank 0's root statistics (what gaz_root_dense hands a caller) as DIR/*.npy")
    args = ap.parse_args()
    if args.moves > 0 and args.steps is not None:
        ap.error("--moves M times M whole moves and replaces --steps; give one of them")
    if args.steps is None:
        args.steps = 40
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if args.impl == "reference":
        return run_reference(args, cfg)
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = load_peaks()
    line = measure(args, cfg, world, rank, local, peaks, want_cpu=(world == 1 and not args.no_cpu_baseline), full=True)
    if args.moves > 0:
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if args.config == "gomoku" and not args.no_extras:
        if world == 1:      # the other BASELINE configurations, short runs, same measurement (driver-visible in the one JSON line)
            subs = {}
            for name in ("connect4", "gumbel", "tictactoe"):
                a2 = argparse.Namespace(**vars(args))
                a2.steps, a2.warmup, a2.games, a2.presearch, a2.config = 20, 3, 0, -1, name
                sub = measure(a2, dict(CONFIGS[name]), world, rank, local, peaks, want_cpu=False, full=False)
                subs[name] = dict(workload=sub["config"]["workload"], value=sub["value"], unit=sub["unit"], ms_per_step=sub["ms_per_step"],
                                  steps=sub["steps"], e2e=sub["e2e"]["value"], positions_per_s=sub["positions_per_s"],
                                  whole_move=sub["whole_move"], sims_per_eval=sub["sims_per_eval"], net_tflops=sub["net_tflops"],
                                  net_frac_of_sustained_peak=sub["net_tflops"] / peaks["sustained"],
                                  roofline=dict((k, sub["roofline"][k]) for k in ("bound", "achieved", "peak", "unit", "frac", "kernel")) if sub["roofline"] else None,
                                  clocks=sub["clocks"], gpu_launches=sub["gpu_launches"])
            # The parity-safe evaluation cache (Session_Cache's role, per-game scope) pays over WHOLE moves - the idle tree of a
            # game re-meets what the other tree evaluated, re-rooted trees re-expand known positions - so it is shown on 8
            # consecutive whole Connect4 moves of every game, with and without it (the headline runs without it).
            pair = {}
            for tag, entries in (("off", 0), ("on", 1 << 23)):
                a3 = argparse.Namespace(**vars(args))
                a3.games, a3.config, a3.eval_cache, a3.moves = 0, "connect4", entries, 8
                sub = measure(a3, dict(CONFIGS["connect4"]), world, rank, local, peaks, want_cpu=False, full=False)
                pair[tag] = dict(value=sub["value"], positions_per_s=sub["positions_per_s"], sims_per_eval=sub["sims_per_eval"],
                                 nn_evals_per_s=sub["nn_evals_per_s"], ms_per_step=sub["ms_per_step"], moves_timed=sub["moves_timed"],
                                 eval_cache=sub["eval_cache"])
            subs["connect4_whole_moves_eval_cache"] = dict(
                workload=CONFIGS["connect4"]["label"] + "; 8 whole moves of every game after one warm-up move; evaluation cache of 2^23 "
                "entries, per-game scope", **pair)
            if rank == 0:
                line["configs"] = subs
        else:               # multi-GPU: a short REAL generation with the NCCL trajectory gather and the writer inside the wall clock
            gen = generation_record(world, rank, local)
            if rank == 0:
                line["e2e_generation"] = gen
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def generation_record(world, rank, local):
    """BASELINE configs[4] in miniature: every rank plays its shard of one generation through the public `run_self_play`
    (Gumbel MCTS n=64 m=16 StableMax on the 10x128+SE network, games cut off after 6 plies so the record stays short), the
    finished trajectories are gathered to rank 0 over NCCL and written with the reference schema by the streaming writer."""
    import shutil
    import tempfile
    import time
    import torch
    import torch.distributed as dist
    from grok_alpha_zero_b200 import games as G
    from grok_alpha_zero_b200.Self_Play import run_self_play
    per_gpu, plies = 4096, 6
    bc = dict(num_resnet_layers=10, num_filters=128, use_stablemax=True, use_se=True)
    tc = dict(MCTS_iteration_limit=64, use_gumbel=True, m=16, c_visit=50.0, c_scale=1.0, max_actions=plies,
              games_per_generation=per_gpu * world, games_per_gpu=per_gpu, num_explore_actions_first=0, num_explore_actions_second=0,
              opening_actions=[[[7, 7], 0.333]])
    folder = tempfile.mkdtemp(prefix="gaz_gen_") if rank == 0 else "/tmp/gaz_gen_unused_%d" % rank
    tm = {}
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    run_self_play(G.Gomoku, (bc, tc, {}), folder, seed=7, timings=tm)
    torch.cuda.synchronize()
    dist.barrier()
    wall = time.perf_counter() - t0
    v = torch.tensor([tm["play_s"], tm["gather_collective_s"], float(tm["gather_bytes"]), float(tm["moves"]), float(tm["sims"])],
                     dtype=torch.float64, device="cuda")
    mx = v.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(v, op=dist.ReduceOp.SUM)
    rec = None
    if rank == 0:
        size = 0
        for f in os.listdir(folder):
            size += os.path.getsize(os.path.join(folder, f))
        shutil.rmtree(folder, ignore_errors=True)
        positions = float(v[3].item())
        rec = dict(what="run_self_play: Gomoku Gumbel n=64 m=16 StableMax, 10x128+SE bf16, %d games/GPU x %d GPUs, games cut off after "
                        "%d plies; NCCL trajectory gather (all_gather of sizes + padded gather to rank 0) and the streaming replay "
                        "writer (8-fold augmentation through gaz_augment on rank 0's GPU) inside the wall clock" % (per_gpu, world, plies),
                   games=per_gpu * world, positions=int(positions), wall_s=wall, positions_per_s=positions / wall,
                   play_s_max=float(mx[0].item()), positions_per_s_search_only=positions / float(mx[0].item()),
                   gather_collective="torch.distributed all_gather + gather (NCCL)", gather_collective_ms=float(mx[1].item()) * 1e3,
                   gather_bytes_total=int(v[2].item()), gather_GBps=float(v[2].item()) / max(float(mx[1].item()), 1e-9) / 1e9,
                   write_s=tm["write_s"], replay_file_bytes=size, datasets_written=int(positions) // plies * 8 * 3,
                   sims=int(v[4].item()))
    return rec


def measure(args, cfg, world, rank, local, peaks, want_cpu, full):
    """one configuration: K timed search rounds (device events), the e2e passes through host buffers, one whole timed move
    (positions/s measured, not derived); returns the JSON line as a dict on every rank (collective reductions inside)"""
    import torch
    import torch.distributed as dist
    n_games = args.games or cfg["games"]

    sb = SelfPlayBench(cfg, n_games, local, noise=not args.no_noise, pool_fraction=args.pool_fraction, eval_cache=args.eval_cache,
                       keep_roots=full and rank == 0 and bool(args.dump_outputs))
    sb.start()
    presearch = 0 if args.moves > 0 else args.presearch
    if presearch < 0:
        presearch = {"gomoku": 232, "connect4": 16, "tictactoe": 12}[cfg["game"]] if cfg["mode"] == "puct" else 20
    done = 0
    while done < presearch:
        n = min(32, presearch - done)
        sb.rounds(n, sync=True)
        done += n
        if sb.run_finished():
            sb.advance_move()

    def barrier():
        sb.eng.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_rounds(k):
        """k search rounds incl. move transitions; returns ms (device events on the engine stream)"""
        sb.eng.timer_begin()
        left = k
        while left > 0:
            n = min(left, 64)
            sb.rounds(n, sync=False)
            left -= n
            if sb.run_finished():  # reads a counter back: synchronises
                sb.advance_move()
        return sb.eng.timer_end()

    def timed_moves(m):
        """m whole moves per game; returns (ms, rounds run)"""
        sb.eng.timer_begin()
        rounds = 0
        for _ in range(m):
            left = cfg["limit"] if cfg["mode"] == "puct" else cfg["limit"] + 17   # Gumbel: + the uncounted root expansions
            while True:
                n = min(64, max(left, 4))
                sb.rounds(n, sync=False)
                rounds += n
                left -= n
                if left <= 0 and sb.run_finished():
                    break
            sb.advance_move()
        return sb.eng.timer_end(), rounds

    if args.moves > 0:
        line = run_moves(args, cfg, sb, timed_moves, barrier, world, rank, local, n_games)
        if full and rank == 0 and args.dump_outputs:
            dump_outputs(sb, args.dump_outputs)
        sb.eng.close()
        sb.net.close()
        del sb
        torch.cuda.empty_cache()
        return line

    # ---- warm-up + timed region -------------------------------------------------------------------
    timed_rounds(args.warmup)
    sims0, evals0, l0 = sb.total_sims(), sb.evals_total(), sb.launches
    sb.net.profile(min(4096, (args.steps + 2) * sb.net.n_conv_tc))
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    ms = timed_rounds(args.steps)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    sims1, evals1, l1 = sb.total_sims(), sb.evals_total(), sb.launches
    sims = sims1 - sims0
    evals = evals1 - evals0
    leaves_per_round = evals / max(1, args.steps)
    roof, conv = dominant_kernel_stats(sb, leaves_per_round, peaks)
    sb.net.profile(0)
    status = sb.eng.status()
    if status != 0:
        raise SystemExit("engine status %d (1 node overflow, 2 slot overflow, 4 LUT miss, 8 bad state)" % status)
    if full and rank == 0 and args.dump_outputs:
        dump_outputs(sb, args.dump_outputs)
        sb.keep_roots = False     # the measurements below copy back only what they need

    # ---- one WHOLE move of every game, timed: fresh start position, the full run (forced root expansions included), root
    # statistics, the tau = 0 move, do_action / check_win, prune_tree of both trees, the next run's begin
    # (skipped with the evaluation cache on: replaying the first move would hit what the timed rounds just stored)
    whole_move, positions_per_s = None, None
    if args.eval_cache == 0:
        sb.alive[:] = True
        sb.next_player[:] = -1
        sb.start()
        m0 = sb.moves
        barrier()
        wm_ms, wm_rounds = timed_moves(1)
        barrier()
        wm = torch.tensor([float(sb.moves - m0)], dtype=torch.float64, device="cuda")
        wmt = torch.tensor([wm_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(wm, op=dist.ReduceOp.SUM)
            dist.all_reduce(wmt, op=dist.ReduceOp.MAX)
        whole_move = dict(moves=int(wm.item()), ms=float(wmt.item()), rounds=int(wm_rounds),
                          what="one whole move of every game from the start position: search run + root statistics + move choice "
                               "+ do_action/check_win + prune_tree (both trees) + next run begin; device events, max over ranks")
        positions_per_s = float(wm.item()) / (float(wmt.item()) * 1e-3)
        if sb.eng.status() != 0:
            raise SystemExit("engine status %d after the whole-move measurement" % sb.eng.status())

    # ---- e2e: host boards in, root statistics out ---------------------------------------------------------
    H, Wd = sb.eng.H, sb.eng.W
    boards = torch.zeros((n_games, H, Wd), dtype=torch.int8).pin_memory().numpy()
    nxt = np.full(n_games, -1, np.int32)
    last = np.full(n_games, -1, np.int32)
    if cfg["opening"] is not None:
        boards.reshape(n_games, -1)[::3, cfg["opening"]] = -1
        nxt[::3] = 1
        last[::3] = cfg["opening"]
    run_mask = np.ones(n_games, np.uint8)
    e2e_ms, e2e_sims = [], 0
    e2e_passes = 2
    for p in range(e2e_passes + 1):
        barrier()
        t0 = time.perf_counter()
        sb.eng.set_games(boards, nxt, last_actions=last)
        sb.next_player = nxt.copy()
        sb.alive[:] = True
        m = np.zeros((n_games, sb.tpg), np.uint8)
        m[np.arange(n_games), 0 if sb.gumbel else (nxt > 0).astype(int)] = 1
        if sb.eng.new_roots(m.reshape(-1)) > 0:
            sb.eng.eval_net()
        sb.eng.expand()
        sb._begin_run()
        sb.rounds(args.steps, sync=False)
        vis, val, info = sb.eng.root_dense(want_values=True)
        barrier()
        dt = (time.perf_counter() - t0) * 1e3
        info = info.reshape(n_games, sb.tpg, 4)
        got = int(info[np.arange(n_games), 0 if sb.gumbel else (nxt > 0).astype(int), 2].sum())
        if p > 0:  # first pass is warm-up
            e2e_ms.append(dt)
            e2e_sims += got
        assert int(vis.sum()) > 0
    h2d = boards.nbytes + n_games * 16 + sb.eng.n_trees * (4 + 1)   # boards + meta + limits + root mask
    if sb.gumbel_noise is not None:
        h2d += sb.eng.n_trees * 256 * 8                              # Gumbel(0,1) root noise table
    d2h = vis.nbytes + val.nbytes + info.nbytes
    e2e_t = torch.tensor([sum(e2e_ms)], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(sims), float(evals), float(e2e_sims), float(sb.moves)], dtype=torch.float64, device="cuda")
    mst = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(mst, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_all = float(mst.item())
    sims_all, evals_all, e2e_sims_all, moves_all = (float(x) for x in tot.tolist())

    if rank == 0:
        value = sims_all / (ms_all * 1e-3)
        e2e_value = e2e_sims_all / (float(e2e_t.item()) * 1e-3)
        line = dict(metric="MCTS simulations/sec", value=value, unit="sims/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms_all / args.steps, higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="bf16", data="synthetic",
                    config=dict(workload=cfg["label"], games_per_gpu=n_games, trees_per_game=sb.tpg,
                                step="one search round = 1 simulation in every running tree (select -> network -> expand/backup)",
                                presearch_rounds=presearch, weights="random-init he_normal, seed 0",
                                l2="per-step working set (%.1f GB of activations + trees) is far larger than the 126 MB L2; no flush needed"
                                   % (sb.net.bytes_allocated() / 1e9),
                                sharding="games by index, no collective on the search path",
                                noise=("none" if not sb.noise else "Gumbel(0,1) on the root logits (host draw, uploaded per move)"
                                       if sb.gumbel else "Dirichlet(alpha=%g, eps=0.25) at every expansion, device Philox "
                                       "streams keyed by global game id (Self_Play.py:38-46)" % cfg["alpha"])),
                    positions_per_s=positions_per_s, whole_move=whole_move,
                    nn_evals_per_s=evals_all / (ms_all * 1e-3), sims_per_eval=sims_all / max(1.0, evals_all),
                    net_tflops=evals_all * sb.flops_per_eval / (ms_all * 1e-3) / 1e12,
                    e2e=dict(value=e2e_value, unit="sims/s", h2d_bytes_per_step=int(h2d / args.steps),
                             d2h_bytes_per_step=int(d2h / args.steps),
                             what="per pass: pinned host boards -> gaz_set_games, fresh roots (1 eval each), %d rounds, "
                                  "gaz_root_dense -> host visit counts/value sums/moves; wall clock incl. copies" % args.steps),
                    gpu_launches=int(l1 - l0), clocks=clocks, roofline=roof,
                    hbm_bytes=dict(engine=sb.eng.bytes_allocated(), net=sb.net.bytes_allocated()),
                    slot_pool=dict(sb.eng.pool_info(), fraction=args.pool_fraction),
                    eval_cache=(dict(sb.eng.eval_cache_stats(), scope="per game",
                                     note="hits are leaf requests served from the table; nn_evals_per_s / net_tflops / sims_per_eval "
                                          "count only what the network evaluated") if args.eval_cache > 0 else None))
        if want_cpu:
            try:
                sys.path.insert(0, os.path.join(ROOT, "oracle"))
                import cpu_selfplay
                cores = os.cpu_count() or 1
                spc = 4
                csteps = 96 if cfg["game"] == "gomoku" else 400   # ~10 s of CPU work on the bounded sample
                r = cpu_selfplay.run_sample(cfg["game"], sb.spec, sb.weights, n_workers=cores, sims_per_step=spc,
                                            steps=csteps, warmup=2, c_puct_init=cfg["c_puct_init"], opening=cfg["opening"],
                                            torch_threads=cores)
                line["cpu_baseline"] = dict(
                    value=r["sims_per_s"], unit="sims/s", cores=cores, kind="port",
                    sample="%d games x %d sims (%d worker threads on the C oracle port of MCTS.py + 1 batching server on the "
                           "fp32 torch-CPU restatement of the network, mean batch %.1f), %.1f s"
                           % (cores, spc * csteps, cores, r["mean_batch"], r["seconds"]))
            except Exception as ex:  # the baseline is a reported number, never a reason to lose the GPU line
                line["cpu_baseline"] = dict(value=None, unit="sims/s", cores=os.cpu_count(), kind="port",
                                            sample="failed: %r" % (ex,))
    sb.eng.close()
    sb.net.close()
    del sb
    torch.cuda.empty_cache()
    return line if rank == 0 else dict(config={}, e2e={}, roofline=None, value=0, unit="", ms_per_step=0, steps=0, positions_per_s=0,
                                       whole_move=None, sims_per_eval=0, net_tflops=0, clocks=None, gpu_launches=0)


if __name__ == "__main__":
    main()
