"""Match vs self-play throughput on one GPU (not a pytest file):
    python tools/arena_bench.py [--games 16384] [--iters 200] [--moves 2] [--reps 2] [--out FILE]
Gomoku 15x15, 10 x 128 + Squeeze-Excitation bf16, `--games` games on one GPU, PUCT with `int(iters * 1.5)` iterations per
move (Self_Play.py:99), no noise, tau = 0.  Alternately, `--reps` times each: a self-play run (one network on both trees of
every game) and a match run (two networks with different weights, each game's trees routed to their own network), each
timing `--moves` whole moves after one warm-up move (which captures the round graph).  Then one more match move with eager
rounds under torch.profiler gives the time of the routing kernels (route_leaves_kernel, route_states_kernel,
scatter_evals_kernel) per network evaluation.  Prints one JSON line with the device name and power limit read in the same
call."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from grok_alpha_zero_b200 import games, netspec  # noqa: E402
from grok_alpha_zero_b200.Self_Play import BatchedSelfPlay  # noqa: E402

ROUTE_KERNELS = ("route_leaves_kernel", "route_states_kernel", "scatter_evals_kernel")


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return dict(name=name, power_limit=power, sm_clock=clock)


def make(args, spec, wa, wb):
    bc = {"use_stablemax": False}
    tc = dict(MCTS_iteration_limit=args.iters, use_gumbel=False, c_puct_init=4.5, max_actions=150,
              num_explore_actions_first=0, num_explore_actions_second=0)
    return BatchedSelfPlay(games.Gomoku, bc, tc, range(args.games), args.games, spec=spec, weights=wa, seed=1,
                           use_noise=False, opponent=None if wb is None else (spec, wb))


def timed(args, spec, wa, wb):
    sp = make(args, spec, wa, wb)
    sp._seat(list(range(sp.n_slots)))
    sp.step()                                  # warm-up move: first eager round, graph capture
    sp.eng.sync()
    s0, m0 = sp.sims, sp.moves
    t0 = time.perf_counter()
    for _ in range(args.moves):
        sp.step()                              # ends with host reads of the root statistics: synchronised
    dt = time.perf_counter() - t0
    rec = dict(seconds=dt, sims_per_s=(sp.sims - s0) / dt, positions_per_s=(sp.moves - m0) / dt,
               ms_per_round=1e3 * dt / (args.moves * sp.limit))
    return sp, rec


def routing_time(sp):
    """one more move with eager rounds (Net.profile switches graph replay off) under torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for n in sp.nets:
        n.profile(1)
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        sp.step()
        sp.eng.sync()
    tot = {k: [0.0, 0] for k in ROUTE_KERNELS}
    for ev in prof.key_averages():
        for k in ROUTE_KERNELS:
            if k in ev.key:
                us = getattr(ev, "self_device_time_total", None)
                tot[k][0] += float(us if us is not None else ev.self_cuda_time_total)
                tot[k][1] += int(ev.count)
    calls = tot["route_leaves_kernel"][1]
    if calls == 0:
        raise RuntimeError("torch.profiler recorded no routing kernel")
    per = {k: tot[k][0] / max(1, tot[k][1]) for k in ROUTE_KERNELS}
    return dict(evaluations=calls, us_per_evaluation=sum(per.values()), us_per_kernel=per)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=200, help="MCTS_iteration_limit (x1.5 per move)")
    ap.add_argument("--moves", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = device_info()
    spec = netspec.build_spec("gomoku", "softmax", num_blocks=10, filters=128, use_se=True)
    wa, wb = netspec.init_weights(spec, seed=1), netspec.init_weights(spec, seed=2)
    runs = {"self_play": [], "match": []}
    route = None
    for rep in range(args.reps):
        for kind, other in (("self_play", None), ("match", wb)):
            sp, rec = timed(args, spec, wa, other)
            runs[kind].append(rec)
            print(kind, rep, json.dumps(rec), flush=True)
            if kind == "match" and rep == args.reps - 1:
                route = routing_time(sp)
            sp.close()
    best = {k: max(r["sims_per_s"] for r in v) for k, v in runs.items()}
    out = dict(tool="arena_bench", game="gomoku", net="10x128+SE bf16", games=args.games, iterations_per_move=int(args.iters * 1.5),
               timed_moves=args.moves, device=dev, self_play=runs["self_play"], match=runs["match"],
               match_over_self_play=best["match"] / best["self_play"],
               match_over_self_play_mean=float(np.mean([r["sims_per_s"] for r in runs["match"]]) /
                                               np.mean([r["sims_per_s"] for r in runs["self_play"]])),
               routing=route)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
