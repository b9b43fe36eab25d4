"""A/B of the evaluation cache (az_set_eval_cache) on the headline workload: 16384 games x 800 simulations, ResNet 4x64 in bf16
(k_resnet_wide).  Both arms play the same seeded games from the same weights; the timed windows alternate off, on, off, on.
Per arm: simulations / s, per simulation step the evaluator rows and the hits / followers the cache served, and k_resnet_wide's
duration inside the timed windows from its device-timer hook (az_resnet_wide_set_timing) set against the rows it computed.
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
from alphazero_implementation_b200 import _lib  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


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
    T_CAP = 1 << 15
    timing = torch.zeros(4 + 2 * T_CAP, dtype=torch.int64, device="cuda")
    timing[4::2] = -1
    _lib.load().az_resnet_wide_set_timing(timing.data_ptr(), T_CAP)  # before any capture: the pointer is baked into the graphs
    arms = {}
    for name, cache in (("off", False), ("on", True)):
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, eval_cache=cache)
        eng = search.engine_for(E, exact=True)
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(1000).random_sample((args.burn_in + args.rounds * K, E))).to(eng.device)
        for i in range(args.burn_in):
            search.simulate_and_move(eng, u[i])
            eng.drain_episodes_device()
        arms[name] = dict(search=search, eng=eng, u=u, next=args.burn_in, windows=[])
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for name in ("off", "on"):
            a = arms[name]
            search, eng = a["search"], a["eng"]
            st0, c0 = eng.stats(), eng.eval_cache_stats()
            launch0 = int(timing[0].item())
            timing[4::2] = -1
            timing[5::2] = 0
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
            st, c = eng.stats(), eng.eval_cache_stats()
            d = {k: st[k] - st0[k] for k in st}
            dc = {k: c[k] - c0[k] for k in c}
            launch1 = int(timing[0].item())
            slots = torch.arange(launch0, launch1, device="cuda") % T_CAP
            dur_ms = (timing[5::2][slots] - timing[4::2][slots]).double() * 1e-6
            sim_steps = K * S
            kern_ms = float(dur_ms.mean().item())
            rows = dc["rows"] / sim_steps
            a["windows"].append({
                "round": r, "sims_per_s": d["simulations"] / ms * 1e3, "ms_per_move_step": ms / K,
                "us_per_sim_step": ms / sim_steps * 1e3,
                "per_sim_step": {"leaves": d["evaluations"] / sim_steps, "rows": rows, "hits": dc["hits"] / sim_steps,
                                 "followers": dc["followers"] / sim_steps, "failed_claims": dc["failed_claims"] / sim_steps,
                                 "evictions": dc["evictions"] / sim_steps},
                "k_resnet_wide": {"launches": launch1 - launch0, "mean_us": kern_ms * 1e3, "min_us": float(dur_ms.min().item()) * 1e3,
                                  "max_us": float(dur_ms.max().item()) * 1e3, "ns_per_row": kern_ms * 1e6 / max(rows, 1e-9),
                                  "share_of_step": kern_ms / (ms / sim_steps)},
            })
    _lib.load().az_resnet_wide_set_timing(None, 0)
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "burn_in": args.burn_in, "steps_per_window": K},
           "card": card(), "cache_log2": arms["on"]["eng"].eval_cache_log2,
           "arms": {n: a["windows"] for n, a in arms.items()}}
    # the evaluator's fixed cost per launch, from the two arms' rows per launch and mean durations (time = fixed + rows * per_row)
    off, on = (np.mean([w["per_sim_step"]["rows"] for w in arms[n]["windows"]]) for n in ("off", "on"))
    t_off, t_on = (np.mean([w["k_resnet_wide"]["mean_us"] for w in arms[n]["windows"]]) for n in ("off", "on"))
    if off > on:
        per_row = (t_off - t_on) / (off - on)
        out["k_resnet_wide_fit"] = {"us_per_row": per_row, "fixed_us_per_launch": t_on - per_row * on,
                                    "fixed_share_on": (t_on - per_row * on) / t_on}
    out["speedup"] = np.mean([w["sims_per_s"] for w in arms["on"]["windows"]]) / np.mean([w["sims_per_s"] for w in arms["off"]["windows"]])
    text = json.dumps(out, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
