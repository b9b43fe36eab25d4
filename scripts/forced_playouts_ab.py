"""A/B of forced playouts and policy target pruning (AlphaZeroSearch(forced_playouts=ForcedPlayouts(k))) on the headline workload:
16384 games x 800 simulations, ResNet 4x64 in bf16 (k_resnet_wide), evaluation cache on.  Arms:
  noise             Dirichlet root noise (alpha 1, fraction 0.25), every search full;
  noise_forced      the same with ForcedPlayouts(2.0): every root child gets about sqrt(2 P N) visits, the targets are pruned;
  noise_cap_forced  the same with the playout cap (160 fast simulations, p_full 0.25): only the full searches are forced.
Same weights and seeds; the timed windows alternate over the arms in one process after an untimed burn-in.  The arms play
different games, so besides the time per move step the output gives what the evaluator does per simulation step (rows computed,
cache hit rate), the share of root selections the forcing rule decided, the visits pruned per forced search (= per recorded
sample), and - from one more search per arm after the windows - the mean entropy of the recorded targets (pruned counts) against
that of the raw visit counts of the same full searches.  Prints one JSON object (and writes it to --out)."""
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


def arm_kwargs(name, k, fast, p_full):
    kw = dict(root_noise=az.RootNoise(alpha=1.0, fraction=0.25, seed=1))
    if "forced" in name:
        kw["forced_playouts"] = az.ForcedPlayouts(k)
    if "cap" in name:
        kw["playout_cap"] = az.PlayoutCap(fast_simulations=fast, full_probability=p_full, seed=1)
    return kw


def entropy(counts):
    c = counts.astype(np.float64)
    p = c / np.maximum(c.sum(1, keepdims=True), 1)
    return float(-(np.where(p > 0, p * np.log(np.where(p > 0, p, 1.0)), 0.0)).sum(1).mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--k", type=float, default=2.0)
    ap.add_argument("--fast-sims", type=int, default=160)
    ap.add_argument("--p-full", type=float, default=0.25)
    ap.add_argument("--burn-in", type=int, default=24, help="untimed move steps per arm (games reach their stationary mix)")
    ap.add_argument("--steps", type=int, default=8, help="move steps per timed window")
    ap.add_argument("--rounds", type=int, default=2, help="windows per arm, alternating over the arms")
    ap.add_argument("--arms", default="noise,noise_forced,noise_cap_forced")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    E, S, K = args.games, args.sims, args.steps
    names = args.arms.split(",")
    arms = {}
    for name in names:
        torch.manual_seed(0)  # the weights bench.py uses
        model = az.ResNet(num_res_blocks=4, num_channels=64)
        search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16,
                                    **arm_kwargs(name, args.k, args.fast_sims, args.p_full))
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
            st0, c0, f0 = eng.stats(), eng.eval_cache_stats(), eng.forced_stats()
            samples = 0
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(K):
                search.simulate_and_move(eng, a["u"][a["next"] + i])
                d = eng.drain_episodes_device()  # the ring holds 2 E + 64 episodes: drained every step, as the generator does
                samples += int(d["s_bb0"].numel())
            ev1.record()
            torch.cuda.synchronize()
            a["next"] += K
            ms = ev0.elapsed_time(ev1)
            st, c, f = eng.stats(), eng.eval_cache_stats(), eng.forced_stats()
            d = {k: st[k] - st0[k] for k in st}
            dc = {k: c[k] - c0[k] for k in c}
            df = {k: f[k] - f0[k] for k in f}
            sim_steps = K * S
            a["windows"].append({
                "round": r, "ms_per_move_step": ms / K, "rows_per_sim_step": dc["rows"] / sim_steps,
                "hit_rate": dc["hits"] / max(d["evaluations"], 1), "sims_per_s": d["simulations"] / ms * 1e3,
                "samples_per_s": samples / ms * 1e3, "forced_selection_share": df["forced_selections"] / max(d["simulations"], 1),
                "pruned_visits_per_forced_search": df["visits_pruned"] / max(df["forced_searches"], 1),
                "zeroed_children_per_forced_search": df["children_zeroed"] / max(df["forced_searches"], 1),
            })
    keys = ("ms_per_move_step", "rows_per_sim_step", "hit_rate", "sims_per_s", "samples_per_s", "forced_selection_share",
            "pruned_visits_per_forced_search", "zeroed_children_per_forced_search")
    mean = {n: {k: float(np.mean([w[k] for w in a["windows"]])) for k in keys} for n, a in arms.items()}
    targets = {}
    for name in names:  # one more search on the current roots: raw counts against the recorded (pruned) targets of full searches
        a = arms[name]
        search, eng = a["search"], a["eng"]
        search.simulate(eng)
        raw = eng.root_stats()["child_N"].cpu().numpy()
        full = eng.search_budgets()[1].cpu().numpy().astype(bool) if eng.playout_cap is not None else np.ones(E, bool)
        rec = eng.policy_targets().cpu().numpy() if eng.forced_playouts is not None else raw
        targets[name] = {"entropy_raw": entropy(raw[full]), "entropy_recorded": entropy(rec[full]), "full_searches": int(full.sum())}
        search.close()
    out = {"workload": {"games": E, "sims": S, "net": "resnet4x64", "dtype": "bf16", "eval_cache": True, "burn_in": args.burn_in,
                        "steps_per_window": K, "k": args.k, "fast_sims": args.fast_sims, "p_full": args.p_full,
                        "noise": {"alpha": 1.0, "fraction": 0.25}},
           "note": "the arms play different games: compare rows per simulation step and hit rates as well as times",
           "card": card(), "arms": {n: a["windows"] for n, a in arms.items()}, "mean": mean, "targets": targets}
    text = json.dumps(out, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
