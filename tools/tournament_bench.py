"""Tournament vs self-play vs sequential matches on one GPU (not a pytest file):
    python tools/tournament_bench.py [--iters 200] [--moves 2] [--reps 2] [--out FILE] [--games-scale 1.0]
Three workloads, each run `--reps` times with the runs alternated, every run timing `--moves` whole moves after one warm-up
move (which captures the round graph); PUCT with `int(iters * 1.5)` iterations per move (Self_Play.py:99), no noise,
tau = 0, every game from the empty board:
  * Gomoku 15x15, 10 x 128 + Squeeze-Excitation bf16: an 8-network round robin of 28 pairs x 584 games (16352 games in one
    batch, the eight networks sharing one activation workspace), self-play of 16352 games with one network, and one pair's
    584-game match alone (the sequential alternative plays 28 of these one after another, at this rate);
  * Connect4, 5 x 128: the same three ways at 28 x 146 = 4088 games;
  * the routing kernels (route_leaves_kernel, route_states_kernel, scatter_evals_kernel) per network evaluation from
    torch.profiler, in separate eager runs (Net.profile switches graph replay off): the Gomoku round robin (K = 8) and a
    Gomoku match of 16384 games (K = 2, the configuration of profiles/arena_bench_gomoku16384.json).
Also reports the device bytes of the round robin's eight networks, against eight networks with a workspace each (computed
from one network's own bytes, not allocated).  Prints one JSON line with the device name, power limit and SM clock read
in the same call.  `--games-scale` shrinks every game count (a quick rehearsal; the published numbers use 1.0)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from grok_alpha_zero_b200 import arena, games, netspec  # noqa: E402
from grok_alpha_zero_b200.Self_Play import BatchedSelfPlay  # noqa: E402
from arena_bench import device_info, routing_time  # noqa: E402  (tools/ is the script's directory)
N_NETS = 8
N_PAIRS = N_NETS * (N_NETS - 1) // 2
WORKLOADS = {
    "gomoku": dict(cls=games.Gomoku, net="10x128+SE bf16", per_pair=584, max_actions=150,
                   spec=dict(num_blocks=10, filters=128, use_se=True)),
    "connect4": dict(cls=games.Connect4, net="5x128 bf16", per_pair=146, max_actions=42,
                     spec=dict(num_blocks=5, filters=128)),
}


def make(args, game, kind, weights, per_pair):
    """kind: "tournament" (8 networks), "self_play" (one network), "match" (one pair) or an int (a match of that many games)"""
    w = WORKLOADS[game]
    spec = netspec.build_spec(game, "softmax", **w["spec"])
    bc = {"use_stablemax": False}
    tc = dict(MCTS_iteration_limit=args.iters, use_gumbel=False, c_puct_init=4.5, max_actions=w["max_actions"],
              num_explore_actions_first=0, num_explore_actions_second=0)
    if kind == "tournament":
        n = N_PAIRS * per_pair
        return BatchedSelfPlay(w["cls"], bc, tc, range(n), n, spec=spec, weights=weights[0], seed=1, use_noise=False,
                               opponents=[(spec, x) for x in weights[1:]],
                               tree_nets=arena.tournament_tree_nets(arena.round_robin(N_NETS), per_pair))
    if kind == "self_play":
        n = N_PAIRS * per_pair
        return BatchedSelfPlay(w["cls"], bc, tc, range(n), n, spec=spec, weights=weights[0], seed=1, use_noise=False)
    n = per_pair if kind == "match" else kind       # an int: a match of that many games
    return BatchedSelfPlay(w["cls"], bc, tc, range(n), n, spec=spec, weights=weights[0], seed=1, use_noise=False,
                           opponent=(spec, weights[1]))


def timed(args, sp):
    sp._seat(list(range(sp.n_slots)))
    sp.step()                                  # warm-up move: first eager round, graph capture
    sp.eng.sync()
    s0, m0 = sp.sims, sp.moves
    t0 = time.perf_counter()
    for _ in range(args.moves):
        sp.step()                              # ends with host reads of the root statistics: synchronised
    dt = time.perf_counter() - t0
    return dict(games=sp.n_slots, seconds=dt, sims_per_s=(sp.sims - s0) / dt, positions_per_s=(sp.moves - m0) / dt,
                ms_per_round=1e3 * dt / (args.moves * sp.limit))


def summary(runs):
    best = {k: max(r["sims_per_s"] for r in v) for k, v in runs.items()}
    mean = {k: float(np.mean([r["sims_per_s"] for r in v])) for k, v in runs.items()}
    return dict(best_sims_per_s=best, mean_sims_per_s=mean,
                tournament_over_self_play=best["tournament"] / best["self_play"],
                tournament_over_sequential_matches=best["tournament"] / best["match"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200, help="MCTS_iteration_limit (x1.5 per move)")
    ap.add_argument("--moves", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--games-scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = device_info()
    out = dict(tool="tournament_bench", nets=N_NETS, pairs=N_PAIRS, iterations_per_move=int(args.iters * 1.5),
               timed_moves=args.moves, device=dev)
    for game, w in WORKLOADS.items():
        per_pair = max(2, int(w["per_pair"] * args.games_scale) // 2 * 2)
        spec = netspec.build_spec(game, "softmax", **w["spec"])
        weights = [netspec.init_weights(spec, seed=s + 1) for s in range(N_NETS)]
        runs = {"tournament": [], "self_play": [], "match": []}
        mem = None
        for rep in range(args.reps):
            for kind in runs:
                sp = make(args, game, kind, weights, per_pair)
                try:
                    if kind == "tournament" and mem is None:
                        own = [n.bytes_allocated() for n in sp.nets]
                        mem = dict(shared_bytes=int(sum(own)), unshared_bytes=int(N_NETS * own[0]),
                                   workspace_bytes=int(own[0] - own[1]), weights_bytes_per_net=int(own[1]))
                    rec = timed(args, sp)
                finally:
                    sp.close()
                runs[kind].append(rec)
                print(game, kind, rep, json.dumps(rec), flush=True)
        out[game] = dict(net=w["net"], games_per_pair=per_pair, games=N_PAIRS * per_pair, runs=runs, memory=mem,
                         **summary(runs))
    per_pair = max(2, int(WORKLOADS["gomoku"]["per_pair"] * args.games_scale) // 2 * 2)
    spec = netspec.build_spec("gomoku", "softmax", **WORKLOADS["gomoku"]["spec"])
    weights = [netspec.init_weights(spec, seed=s + 1) for s in range(N_NETS)]
    route = {}
    for label, kind in (("k8", "tournament"), ("k2", max(2, int(16384 * args.games_scale) // 2 * 2))):
        sp = make(args, "gomoku", kind, weights, per_pair)
        try:
            sp._seat(list(range(sp.n_slots)))
            route[label] = dict(nets=len(sp.nets), games=sp.n_slots, **routing_time(sp))
        finally:
            sp.close()
        print("routing", label, json.dumps(route[label]), flush=True)
    out["routing"] = route
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
