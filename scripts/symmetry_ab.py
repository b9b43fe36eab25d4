"""A/B of symmetric leaf evaluation (AlphaZeroSearch(symmetric=True)) on the headline workload: 16384 games x 800 simulations,
ResNet 4x64 in bf16 (k_resnet_wide), evaluation cache on.  Arm "off" is the plain search; arm "on" evaluates every leaf in its
canonical orientation under the left-right mirror.  Both arms start from the same weights and seeds; the timed windows alternate
off, on, off, on in one process after an untimed burn-in.
The arms play different games (f_sym != f), so besides simulations / s the output compares what the evaluator does per simulation
step: rows computed, cache hit and follower rates, and k_resnet_wide's in-region time per computed row (az_resnet_wide_set_timing).
For arm "on", one further untimed move step counts the share of the evaluated leaves that were mirrored.
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
from alphazero_implementation_b200.engine import LEAF_EVAL, LEAF_SERVED, POLICY_LOGITS  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def mirrored_share(search, eng, u):
    """one move step driven simulation by simulation (un-graphed, same kernels): mirrored / all non-terminal leaves"""
    g = search._graphed
    n = eng.n_active
    live = mirrored = 0
    eng.select_leaves()
    for i in range(search.num_simulations):
        st = eng.leaf_info()["status"]
        ok = (st == LEAF_EVAL) | (st == LEAF_SERVED)
        live += int(ok.sum())
        mirrored += int((eng.leaf_mirror()[:n].bool() & ok).sum())
        logits, values = g.evaluate()
        if i + 1 < search.num_simulations:
            eng.expand_backup_select(logits, values, POLICY_LOGITS)
        else:
            eng.expand_backup(logits, values, POLICY_LOGITS)
    eng.sample_moves(u)
    return {"leaves": live, "mirrored": mirrored, "share": mirrored / max(live, 1)}


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
    for name in ("off", "on"):
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, symmetric=name == "on")
        eng = search.engine_for(E, exact=True)
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(1000).random_sample((args.burn_in + args.rounds * K + 1, E))).to(eng.device)
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
            leaves = max(d["evaluations"], 1)
            rows = dc["rows"] / sim_steps
            kern_ms = float(dur_ms.mean().item())
            a["windows"].append({
                "round": r, "sims_per_s": d["simulations"] / ms * 1e3, "ms_per_move_step": ms / K,
                "per_sim_step": {"leaves": d["evaluations"] / sim_steps, "rows": rows, "hits": dc["hits"] / sim_steps,
                                 "followers": dc["followers"] / sim_steps, "failed_claims": dc["failed_claims"] / sim_steps},
                "hit_rate": dc["hits"] / leaves, "follower_rate": dc["followers"] / leaves, "rows_per_leaf": dc["rows"] / leaves,
                "k_resnet_wide": {"launches": launch1 - launch0, "mean_us": kern_ms * 1e3, "ns_per_row": kern_ms * 1e6 / max(rows, 1e-9)},
            })
    _lib.load().az_resnet_wide_set_timing(None, 0)
    on = arms["on"]
    share = mirrored_share(on["search"], on["eng"], on["u"][on["next"]])
    mean = {n: {k: float(np.mean([w[k] for w in a["windows"]])) for k in ("sims_per_s", "ms_per_move_step", "hit_rate", "follower_rate")}
            for n, a in arms.items()}
    for n, a in arms.items():
        mean[n]["rows_per_sim_step"] = float(np.mean([w["per_sim_step"]["rows"] for w in a["windows"]]))
        mean[n]["ns_per_row"] = float(np.mean([w["k_resnet_wide"]["ns_per_row"] for w in a["windows"]]))
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "eval_cache": True, "burn_in": args.burn_in,
                        "steps_per_window": K},
           "note": "the arms play different games (f_sym != f): compare rows, hit rates and cost per row as well as sims/s",
           "card": card(), "cache_log2": on["eng"].eval_cache_log2, "mirrored_leaves_on": share,
           "arms": {n: a["windows"] for n, a in arms.items()}, "mean": mean,
           "on_over_off_sims_per_s": mean["on"]["sims_per_s"] / mean["off"]["sims_per_s"]}
    text = json.dumps(out, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
