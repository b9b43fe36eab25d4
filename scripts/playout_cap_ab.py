"""A/B of playout cap randomization (AlphaZeroSearch(playout_cap=PlayoutCap(...))) on the headline workload: 16384 games x 800
simulations, ResNet 4x64 in bf16 (k_resnet_wide), evaluation cache on.  Arms:
  off          every search runs 800 new simulations on a fresh root (the reference's self-play);
  cap          fast_sims = 160, p_full = 0.25: a quarter of the searches are full and recorded, the rest only pick the move;
  reuse        subtree reuse (max_root_visits 4 S), every search runs 800 new simulations;
  reuse_budget subtree reuse with the total-visit budget (p_full = 1, visit_budget): a search tops the root up to 800 visits.
Same weights and seeds; the timed windows alternate over the arms in one process after an untimed burn-in.  The arms play
different games, so besides the time per move step the output gives what the evaluator does per simulation step (rows computed,
cache hit rate) and the rates users pay for: moves, finished games and recorded training samples per second, and the mean number of
new simulations per search.  Prints one JSON object (and writes it to --out)."""
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


def arm_kwargs(name, S, fast, p_full):
    if name == "cap":
        return dict(playout_cap=az.PlayoutCap(fast_simulations=fast, full_probability=p_full, seed=1))
    if name == "reuse":
        return dict(subtree_reuse=True)
    if name == "reuse_budget":
        return dict(subtree_reuse=True, playout_cap=az.PlayoutCap(fast_simulations=S, full_probability=1.0, visit_budget=True))
    return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--fast-sims", type=int, default=160)
    ap.add_argument("--p-full", type=float, default=0.25)
    ap.add_argument("--burn-in", type=int, default=24, help="untimed move steps per arm (games reach their stationary mix)")
    ap.add_argument("--steps", type=int, default=8, help="move steps per timed window")
    ap.add_argument("--rounds", type=int, default=2, help="windows per arm, alternating over the arms")
    ap.add_argument("--arms", default="off,cap,reuse,reuse_budget")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    E, S, K = args.games, args.sims, args.steps
    names = args.arms.split(",")
    arms = {}
    for name in names:
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, **arm_kwargs(name, S, args.fast_sims, args.p_full))
        eng = search.engine_for(E, exact=True)
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(1000).random_sample((args.burn_in + args.rounds * K, E))).to(eng.device)
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
            games = samples = 0
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(K):
                search.simulate_and_move(eng, a["u"][a["next"] + i])
                d = eng.drain_episodes_device()  # the ring holds 2 E + 64 episodes: drained every step, as the generator does
                games += int(d["ep_slot"].numel())
                samples += int(d["s_bb0"].numel())
            ev1.record()
            torch.cuda.synchronize()
            a["next"] += K
            ms = ev0.elapsed_time(ev1)
            st, c = eng.stats(), eng.eval_cache_stats()
            d = {k: st[k] - st0[k] for k in st}
            dc = {k: c[k] - c0[k] for k in c}
            sim_steps = K * S
            a["windows"].append({
                "round": r, "ms_per_move_step": ms / K, "rows_per_sim_step": dc["rows"] / sim_steps,
                "leaves_per_sim_step": d["evaluations"] / sim_steps, "hit_rate": dc["hits"] / max(d["evaluations"], 1),
                "moves_per_s": d["moves"] / ms * 1e3, "games_per_s": games / ms * 1e3, "samples_per_s": samples / ms * 1e3,
                "new_sims_per_search": d["simulations"] / max(d["moves"], 1), "sims_per_s": d["simulations"] / ms * 1e3,
            })
    keys = ("ms_per_move_step", "rows_per_sim_step", "hit_rate", "moves_per_s", "games_per_s", "samples_per_s", "new_sims_per_search",
            "sims_per_s")
    mean = {n: {k: float(np.mean([w[k] for w in a["windows"]])) for k in keys} for n, a in arms.items()}
    base = mean.get("off")
    ratios = {n: {k: m[k] / base[k] for k in ("ms_per_move_step", "games_per_s", "samples_per_s")} for n, m in mean.items()} if base else {}
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "eval_cache": True, "burn_in": args.burn_in,
                        "steps_per_window": K, "fast_sims": args.fast_sims, "p_full": args.p_full},
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
