"""A/B of AlphaZero's self-play exploration on the headline workload: 16384 games x 800 simulations, ResNet 4x64 in bf16
(k_resnet_wide), evaluation cache on.  Arm "off" is the reference's self-play; arm "on" adds Dirichlet noise on the root priors
(alpha 1.0, fraction 0.25) and the greedy cutoff at ply 12.  Both arms play seeded games from the same weights; the timed
windows alternate off, on, off, on in one process.
Per arm: simulations / s, per simulation step the evaluator rows and the cache's hit and follower rates, and the diversity of the
games: distinct positions among the finished episodes' samples at plies 6, 10 and 14.  Separately, k_root_noise's own time
(CUDA events around the launch, 16384 roots with 7 legal columns) against the measured move step.
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

PLIES = (6, 10, 14)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def diversity(drains):
    """distinct / total positions at each ply in PLIES over the finished episodes of `drains` (device dicts of
    Engine.drain_episodes_device)."""
    seen = {p: set() for p in PLIES}
    total = {p: 0 for p in PLIES}
    for d in drains:
        ln, off = d["ep_len"].cpu().numpy(), d["ep_offset"].cpu().numpy()
        b0, b1 = d["s_bb0"].cpu().numpy(), d["s_bb1"].cpu().numpy()
        for p in PLIES:
            has = ln > p
            idx = off[has] + p
            total[p] += int(has.sum())
            seen[p].update(zip(b0[idx].tolist(), b1[idx].tolist()))
    return {f"ply{p}": {"samples": total[p], "distinct": len(seen[p]), "distinct_share": len(seen[p]) / max(total[p], 1)}
            for p in PLIES}


def noise_kernel_us(E, reps=50):
    """k_root_noise alone: CUDA events around az_apply_root_noise on E fresh roots at the initial position (7 legal columns)."""
    eng = az.Engine(num_games=E, num_simulations=2)
    eng.set_root_noise(1.0, 0.25, 0)
    z = np.zeros(E, np.uint64)
    times = []
    for i in range(reps + 5):
        eng.set_roots(z, z, np.zeros(E, np.uint8))
        eng.run_simulations(1, 1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.apply_root_noise()
        b.record()
        torch.cuda.synchronize()
        if i >= 5:
            times.append(a.elapsed_time(b) * 1e3)
    eng.close()
    return {"trees": E, "mean_us": float(np.mean(times)), "min_us": float(np.min(times)), "max_us": float(np.max(times))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--burn-in", type=int, default=24, help="untimed move steps per arm (games reach their stationary mix)")
    ap.add_argument("--steps", type=int, default=8, help="move steps per timed window")
    ap.add_argument("--rounds", type=int, default=2, help="windows per arm, alternating off / on")
    ap.add_argument("--alpha", type=float, default=1.0)
    ap.add_argument("--fraction", type=float, default=0.25)
    ap.add_argument("--sampling-moves", type=int, default=12)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    E, S, K = args.games, args.sims, args.steps
    arms = {}
    for name in ("off", "on"):
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        noise = az.RootNoise(alpha=args.alpha, fraction=args.fraction, seed=0) if name == "on" else None
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, root_noise=noise)
        eng = search.engine_for(E, exact=True)
        eng.reset_games()
        eng.set_greedy_from(args.sampling_moves if name == "on" else None)
        u = torch.from_numpy(np.random.RandomState(1000).random_sample((args.burn_in + args.rounds * K, E))).to(eng.device)
        for i in range(args.burn_in):
            search.simulate_and_move(eng, u[i])
            eng.drain_episodes_device()
        arms[name] = dict(search=search, eng=eng, u=u, next=args.burn_in, windows=[], drains=[])
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for name in ("off", "on"):
            a = arms[name]
            search, eng = a["search"], a["eng"]
            st0, c0 = eng.stats(), eng.eval_cache_stats()
            n0 = eng.launch_count
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(K):
                search.simulate_and_move(eng, a["u"][a["next"] + i])
                if i % 8 == 7 or i + 1 == K:
                    a["drains"].append(eng.drain_episodes_device())
            ev1.record()
            torch.cuda.synchronize()
            a["next"] += K
            ms = ev0.elapsed_time(ev1)
            st, c = eng.stats(), eng.eval_cache_stats()
            d = {k: st[k] - st0[k] for k in st}
            dc = {k: c[k] - c0[k] for k in c}
            sim_steps = K * S
            leaves = max(d["evaluations"], 1)
            a["windows"].append({
                "round": r, "sims_per_s": d["simulations"] / ms * 1e3, "ms_per_move_step": ms / K,
                "engine_launches_per_move_step": (eng.launch_count - n0) / K,
                "per_sim_step": {"leaves": d["evaluations"] / sim_steps, "rows": dc["rows"] / sim_steps, "hits": dc["hits"] / sim_steps,
                                 "followers": dc["followers"] / sim_steps},
                "hit_rate": dc["hits"] / leaves, "follower_rate": dc["followers"] / leaves,
            })
    step_ms = float(np.mean([w["ms_per_move_step"] for w in arms["on"]["windows"]]))
    kern = noise_kernel_us(E)
    kern["share_of_move_step"] = kern["mean_us"] * 1e-3 / step_ms
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "eval_cache": True, "burn_in": args.burn_in,
                        "steps_per_window": K, "noise": {"alpha": args.alpha, "fraction": args.fraction,
                                                         "sampling_moves": args.sampling_moves}},
           "card": card(), "k_root_noise": kern,
           "arms": {n: {"windows": a["windows"], "diversity": diversity(a["drains"]),
                        "sims_per_s_mean": float(np.mean([w["sims_per_s"] for w in a["windows"]]))} for n, a in arms.items()}}
    out["on_over_off"] = out["arms"]["on"]["sims_per_s_mean"] / out["arms"]["off"]["sims_per_s_mean"]
    text = json.dumps(out, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
