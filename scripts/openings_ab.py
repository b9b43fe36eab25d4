"""A/B of opening positions (Engine.set_openings / EpisodeGenerator(openings=)) on the headline workload: 16384 games x 800
simulations, ResNet 4x64 in bf16 (k_resnet_wide), evaluation cache on.  Arms:
  off     every game starts from the empty board (the reference's self-play);
  plies   Openings(min_plies=0, max_plies=4): the empty board and 0 to 4 random plies that neither win nor fill the board;
  set256  256 distinct 6-ply openings (distinct_openings, distinct up to the mirror), each game starts from one of them.
Same weights and seeds; the timed windows alternate over the arms in one process after an untimed burn-in.  More diverse games are
expected to lower the cache hit rate and so raise the cost of a move step: per window the output gives the distinct positions among
the recorded samples, the distinct games (sample sequences), the cache hit rate and evaluator rows per simulation step, ms per move
step and the mean game length (searched plies).  k_openings' device time per move step comes from one torch.profiler run per arm
with openings, after the timed windows.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alphazero_implementation_b200 as az  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def arm_openings(name):
    if name == "plies":
        return az.Openings(min_plies=0, max_plies=4, seed=1)
    if name == "set256":
        return az.Openings(positions=az.distinct_openings(256, 6, seed=2), seed=1)
    return None


def diversity(batches):
    """distinct (bb0, bb1) among the samples, distinct games (their sample sequences), games, samples"""
    pos, games = set(), set()
    n_games = n_samples = 0
    for d in batches:
        b0, b1 = d["s_bb0"].cpu().numpy(), d["s_bb1"].cpu().numpy()
        ln, off = d["ep_len"].cpu().numpy(), d["ep_offset"].cpu().numpy()
        pos.update(zip(b0.tolist(), b1.tolist()))
        for o, n in zip(off.tolist(), ln.tolist()):
            games.add(b0[o:o + n].tobytes() + b1[o:o + n].tobytes())
        n_games += len(ln)
        n_samples += len(b0)
    return len(pos), len(games), n_games, n_samples


def k_openings_ms(search, eng, u, steps):
    """device time of k_openings per move step over `steps` move steps (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            search.simulate_and_move(eng, u[i])
            eng.drain_episodes_device()
        torch.cuda.synchronize()
    us = 0.0
    for e in prof.key_averages():
        if "k_openings" in e.key:
            us += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return us / 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--burn-in", type=int, default=24, help="untimed move steps per arm (games reach their stationary mix)")
    ap.add_argument("--steps", type=int, default=8, help="move steps per timed window")
    ap.add_argument("--rounds", type=int, default=2, help="windows per arm, alternating over the arms")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--arms", default="off,plies,set256")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    E, S, K = args.games, args.sims, args.steps
    names = args.arms.split(",")
    arms = {}
    n_u = args.burn_in + args.rounds * K + args.profile_steps
    for name in names:
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16)
        eng = search.engine_for(E, exact=True)
        eng.set_openings(arm_openings(name))
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(1000).random_sample((n_u, E))).to(eng.device)
        for i in range(args.burn_in):
            search.simulate_and_move(eng, u[i])
            eng.drain_episodes_device()
        arms[name] = dict(search=search, eng=eng, u=u, next=args.burn_in, windows=[])
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for name in names:
            a = arms[name]
            search, eng = a["search"], a["eng"]
            st0, c0 = eng.stats(), eng.eval_cache_stats()
            batches = []
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(K):
                search.simulate_and_move(eng, a["u"][a["next"] + i])
                batches.append(eng.drain_episodes_device())  # the ring holds 2 E + 64 episodes: drained every step
            ev1.record()
            torch.cuda.synchronize()
            a["next"] += K
            ms = ev0.elapsed_time(ev1)
            st, c = eng.stats(), eng.eval_cache_stats()
            d = {k: st[k] - st0[k] for k in st}
            dc = {k: c[k] - c0[k] for k in c}
            npos, ngames, n_ep, n_s = diversity(batches)
            a["windows"].append({
                "round": r, "ms_per_move_step": ms / K, "rows_per_sim_step": dc["rows"] / (K * S),
                "hit_rate": dc["hits"] / max(d["evaluations"], 1), "distinct_positions": npos, "distinct_games": ngames, "games": n_ep,
                "samples": n_s, "mean_game_length": n_s / max(n_ep, 1), "sims_per_s": d["simulations"] / ms * 1e3,
            })
    for name in names:
        a = arms[name]
        if a["eng"].openings is not None:
            a["k_openings_ms_per_move_step"] = k_openings_ms(a["search"], a["eng"], a["u"][a["next"]:], args.profile_steps)
    keys = ("ms_per_move_step", "rows_per_sim_step", "hit_rate", "distinct_positions", "distinct_games", "games", "mean_game_length",
            "sims_per_s")
    mean = {n: {k: float(np.mean([w[k] for w in a["windows"]])) for k in keys} for n, a in arms.items()}
    for n, a in arms.items():
        if "k_openings_ms_per_move_step" in a:
            mean[n]["k_openings_ms_per_move_step"] = a["k_openings_ms_per_move_step"]
    base = mean.get("off")
    ratios = {n: {k: m[k] / base[k] for k in ("ms_per_move_step", "rows_per_sim_step", "distinct_positions")} for n, m in mean.items()} if base else {}
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "eval_cache": True, "burn_in": args.burn_in,
                        "steps_per_window": K},
           "note": "the arms play different games: compare rows per simulation step and hit rates as well as times",
           "card": card(), "arms": {n: a["windows"] for n, a in arms.items()}, "mean": mean, "over_off": ratios}
    text = json.dumps(out, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
