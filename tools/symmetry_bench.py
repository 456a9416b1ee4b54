"""Cost of symmetric network evaluation on one GPU (not a pytest file):
    python tools/symmetry_bench.py [--game gomoku|connect4|all] [--iters 150] [--moves 2] [--reps 2] [--games-scale 1.0]
                                   [--out FILE]
Self-play with eval_symmetry "none" / "random" / "ensemble", the three modes alternated `--reps` times, every run timing
`--moves` whole moves after one warm-up move (which captures the round graph); PUCT with `int(iters * 1.5)` iterations
per move (Self_Play.py:99; 225 for Gomoku by default: a limit below the 225 legal moves of the empty board would
become 3 x 225 by the 3 * n_legal rule of MCTS.py:543-546), no noise, tau = 0, every game from the empty board, all games resident:
  * Gomoku 15x15, 10 x 128 + Squeeze-Excitation bf16, 16384 games (n = 8 symmetries);
  * Connect4, 5 x 128, 4096 games (n = 2).
Reports simulations/s and ms per round, and the pack and scatter kernels (sym_states_kernel, sym_scatter_kernel) and the
leaf routing kernel per evaluation from torch.profiler in a separate eager run (Net.profile switches graph replay off) of
8 search rounds per mode.  Prints one JSON line with the device name, power limit and SM clock read in the same call.
`--games-scale` shrinks the game counts (a quick rehearsal; published numbers use 1.0)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from grok_alpha_zero_b200 import games, netspec  # noqa: E402
from grok_alpha_zero_b200.Self_Play import BatchedSelfPlay  # noqa: E402
from arena_bench import device_info  # noqa: E402  (tools/ is the script's directory)

MODES = ("none", "random", "ensemble")
SYM_KERNELS = ("route_leaves_kernel", "sym_states_kernel", "sym_scatter_kernel")
WORKLOADS = {
    "gomoku": dict(cls=games.Gomoku, net="10x128+SE bf16", games=16384, max_actions=150, n_sym=8,
                   spec=dict(num_blocks=10, filters=128, use_se=True)),
    "connect4": dict(cls=games.Connect4, net="5x128 bf16", games=4096, max_actions=42, n_sym=2,
                     spec=dict(num_blocks=5, filters=128)),
}


def make(game, mode, iters, n_games, weights):
    w = WORKLOADS[game]
    spec = netspec.build_spec(game, "softmax", **w["spec"])
    tc = dict(MCTS_iteration_limit=iters, use_gumbel=False, c_puct_init=4.5, max_actions=w["max_actions"],
              num_explore_actions_first=0, num_explore_actions_second=0, eval_symmetry=mode)
    return BatchedSelfPlay(w["cls"], {"use_stablemax": False}, tc, range(n_games), n_games, spec=spec, weights=weights,
                           seed=1, use_noise=False)


def timed(args, sp):
    sp._seat(list(range(sp.n_slots)))
    sp.step()                                  # warm-up move: first eager round, graph capture
    sp.eng.sync()
    s0 = sp.sims
    t0 = time.perf_counter()
    for _ in range(args.moves):
        sp.step()                              # ends with host reads of the root statistics: synchronised
    dt = time.perf_counter() - t0
    return dict(seconds=dt, sims_per_s=(sp.sims - s0) / dt, ms_per_round=1e3 * dt / (args.moves * sp.limit))


def kernel_time(sp):
    """8 eager search rounds under torch.profiler: microseconds per evaluation of each symmetry kernel"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for n in sp.nets:
        n.profile(1)
    torch.cuda.init()
    sp._seat(list(range(sp.n_slots)))
    sp.eng.sync()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        sp.eng.run_begin(sp.limit)
        sp.eng.rounds_net(8)
    tot = {k: [0.0, 0] for k in SYM_KERNELS}
    for ev in prof.key_averages():
        for k in SYM_KERNELS:
            if k in ev.key:
                us = getattr(ev, "self_device_time_total", None)
                tot[k][0] += float(us if us is not None else ev.self_cuda_time_total)
                tot[k][1] += int(ev.count)
    calls = tot["sym_states_kernel"][1]
    if calls == 0:
        raise RuntimeError("torch.profiler recorded no symmetry kernel")
    per = {k: tot[k][0] / max(1, tot[k][1]) for k in SYM_KERNELS}
    return dict(evaluations=calls, us_per_evaluation=sum(per.values()), us_per_kernel=per)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--game", choices=("gomoku", "connect4", "all"), default="all")
    ap.add_argument("--iters", type=int, default=150, help="MCTS_iteration_limit (x1.5 per move)")
    ap.add_argument("--moves", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--games-scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    out = dict(tool="symmetry_bench", iterations_per_move=int(args.iters * 1.5), timed_moves=args.moves, device=device_info())
    for game, w in WORKLOADS.items():
        if args.game not in ("all", game):
            continue
        n_games = max(2, int(w["games"] * args.games_scale))
        weights = netspec.init_weights(netspec.build_spec(game, "softmax", **w["spec"]), seed=1)
        runs = {m: [] for m in MODES}
        for rep in range(args.reps):
            for mode in MODES:
                sp = make(game, mode, args.iters, n_games, weights)
                try:
                    runs[mode].append(timed(args, sp))
                finally:
                    sp.close()
                print(game, mode, rep, json.dumps(runs[mode][-1]), flush=True)
        kernels = {}
        for mode in MODES[1:]:
            sp = make(game, mode, args.iters, n_games, weights)
            try:
                kernels[mode] = kernel_time(sp)
            finally:
                sp.close()
            print(game, mode, "kernels", json.dumps(kernels[mode]), flush=True)
        best = {m: max(r["sims_per_s"] for r in v) for m, v in runs.items()}
        out[game] = dict(net=w["net"], games=n_games, n_sym=w["n_sym"], runs=runs, best_sims_per_s=best,
                         mean_sims_per_s={m: float(np.mean([r["sims_per_s"] for r in v])) for m, v in runs.items()},
                         random_over_none=best["random"] / best["none"], ensemble_over_none=best["ensemble"] / best["none"],
                         kernels=kernels)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
