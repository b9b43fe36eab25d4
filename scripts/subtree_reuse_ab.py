"""A/B of subtree reuse (AlphaZeroSearch(subtree_reuse=True): max_root_visits V = 4 S) on the headline workload: 16384 games x
800 simulations, ResNet 4x64 in bf16 (k_resnet_wide), evaluation cache on.  Arm "off" starts every move step's search from a fresh
root; arm "on" keeps the played child's subtree.  Both arms run S new simulations per move step, from the same weights and seeds;
the timed windows alternate off, on, off, on in one process after an untimed burn-in.
The arms play different games (a root with more visits samples other moves), so besides simulations / s the output compares what
the evaluator does per simulation step (rows computed, cache hit rate), the mean root visits at search start, the retained / fresh
/ dropped shares of the moves, the arena's device bytes, and k_reroot's device time per move step (one extra move step of arm "on"
under torch.profiler) with the bytes the compaction has to move (W and M of every retained node, read and written) over that time.
Prints one JSON object (and writes it to --out)."""
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


def reroot_profile(search, eng, u):
    """device time of k_reroot and k_sample_moves in one move step, and the retained nodes it moved"""
    r0 = eng.reuse_stats()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        search.simulate_and_move(eng, u)
        torch.cuda.synchronize()
    r1 = eng.reuse_stats()
    us = {"k_reroot": 0.0, "k_sample_moves": 0.0}
    for ev in prof.events():
        for k in us:
            if k in ev.name:
                us[k] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    nodes = r1["nodes"] - r0["nodes"]
    moved = nodes * 2 * (8 + 16)  # W (f64) and M (16 B) of every retained node, read once and written once
    return {"k_reroot_us": us["k_reroot"], "k_sample_moves_us": us["k_sample_moves"], "retained_nodes": nodes,
            "moved_bytes": moved, "moved_GB_per_s": moved / max(us["k_reroot"], 1e-9) * 1e-3,
            "moves": {k: r1[k] - r0[k] for k in ("retained", "fresh", "dropped")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--burn-in", type=int, default=24, help="untimed move steps per arm (games reach their stationary mix)")
    ap.add_argument("--steps", type=int, default=8, help="move steps per timed window")
    ap.add_argument("--rounds", type=int, default=2, help="windows per arm, alternating off / on")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    E, S, K = args.games, args.sims, args.steps
    arms = {}
    for name in ("off", "on"):
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, subtree_reuse=name == "on")
        eng = search.engine_for(E, exact=True)
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(1000).random_sample((args.burn_in + args.rounds * K + 1, E))).to(eng.device)
        for i in range(args.burn_in):
            search.simulate_and_move(eng, u[i])
            eng.drain_episodes_device()
        arms[name] = dict(search=search, eng=eng, u=u, next=args.burn_in, windows=[], device_bytes=eng.device_bytes,
                          tree_capacity=eng.tree_capacity)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for name in ("off", "on"):
            a = arms[name]
            search, eng = a["search"], a["eng"]
            st0, c0, r0 = eng.stats(), eng.eval_cache_stats(), eng.reuse_stats()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(K):
                search.simulate_and_move(eng, a["u"][a["next"] + i])
                if i % 8 == 7 or i + 1 == K:
                    eng.drain_episodes_device()
            ev1.record()
            torch.cuda.synchronize()
            a["next"] += K
            ms = ev0.elapsed_time(ev1)
            st, c, rs = eng.stats(), eng.eval_cache_stats(), eng.reuse_stats()
            d = {k: st[k] - st0[k] for k in st}
            dc = {k: c[k] - c0[k] for k in c}
            dr = {k: rs[k] - r0[k] for k in rs}
            moves = max(d["moves"], 1)
            sim_steps = K * S
            a["windows"].append({
                "round": r, "sims_per_s": d["simulations"] / ms * 1e3, "ms_per_move_step": ms / K,
                "rows_per_sim_step": dc["rows"] / sim_steps, "leaves_per_sim_step": d["evaluations"] / sim_steps,
                "hit_rate": dc["hits"] / max(d["evaluations"], 1), "follower_rate": dc["followers"] / max(d["evaluations"], 1),
                # a retained root starts with N(c) visits, a fresh one with 0 (moves that ended a game start a fresh root, too)
                "mean_root_visits_at_search_start": dr["visits"] / moves,
                "shares": {k: dr[k] / moves for k in ("retained", "fresh", "dropped")},
                "retained_nodes_per_retained_move": dr["nodes"] / max(dr["retained"], 1),
            })
    on = arms["on"]
    prof = reroot_profile(on["search"], on["eng"], on["u"][on["next"]])
    prof["share_of_move_step"] = prof["k_reroot_us"] * 1e-3 / float(np.mean([w["ms_per_move_step"] for w in on["windows"]]))
    keys = ("sims_per_s", "ms_per_move_step", "rows_per_sim_step", "hit_rate", "mean_root_visits_at_search_start")
    mean = {n: {k: float(np.mean([w[k] for w in a["windows"]])) for k in keys} for n, a in arms.items()}
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "eval_cache": True, "burn_in": args.burn_in,
                        "steps_per_window": K, "max_root_visits_on": on["search"].max_root_visits},
           "note": "the arms play different games: compare rows per simulation step and hit rates as well as sims/s",
           "card": card(), "arena": {n: {"device_bytes": a["device_bytes"], "tree_capacity": a["tree_capacity"]} for n, a in arms.items()},
           "k_reroot": prof, "arms": {n: a["windows"] for n, a in arms.items()}, "mean": mean,
           "on_over_off_sims_per_s": mean["on"]["sims_per_s"] / mean["off"]["sims_per_s"]}
    text = json.dumps(out, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
