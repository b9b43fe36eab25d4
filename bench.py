#!/usr/bin/env python
"""Headline benchmark: MCTS simulations/s (and self-play games/s) for Connect4 self-play on B200, network in the loop.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload.  N = 1: BASELINE.json configs[2] — 16384 concurrent games x 800 simulations/move with a bf16 ResNet-style
policy/value net (4 residual blocks x 64 channels, random init, 25.3 MFLOP per position) in the loop: every simulation step
is one evaluator launch over the leaves that wait for an evaluation (`k_resnet_wide`, hand-written tcgen05, leaf gather + heads
fused) and one tree launch (`k_expand_select`: expansion + backup, the next selection, and the list of the leaves to evaluate).  N > 1: configs[3] — 65536 games sharded over the ranks (65536 / N per GPU, "strong" split of the
fixed total), and the episodes finished in the timed region are all-gathered over NCCL INSIDE the timed region.
One STEP = one move step of the self-play loop for every game (episode_generator.py:48-78): 800 simulations per tree, then the
move (`az_sample_moves`: record the samples, draw the moves, recycle finished games).

`value`   device-resident: the steps' uniforms are already in HBM, one CUDA-event pair around the K timed steps, max over
          ranks.  `burn-in` untimed move steps come first so that the timed steps see the stationary mix of a running
          self-play loop (games at every stage, finishing and restarting), not the opening all games share after a reset.
          No L2 flush: one step streams the 2.2 GB tree arena (16384 trees x 5608 nodes x 24 B) 800 times, far beyond the 126 MB L2.
`e2e`     the public API (`EpisodeGenerator.iter_steps`) continuing the same games: per step the uniforms come from pinned host
          memory and the finished episodes + ring counters are read back to pinned host memory (N > 1: plus the all-gather).
`roofline` of the dominant kernel (`k_resnet_wide`, tensor-bound): algorithmic FLOPs per launch (evaluated leaves x FLOPs per
          position) / the kernel's mean duration, CUDA events around every one of its 800 launches in one extra un-graphed move
          step right after the timed region, against the measured sustained bf16 rate of MEASURED_PEAKS.json.
`--impl reference`  the CPU arm: the reference algorithm (oracle/c4_oracle.c, the C restatement pinned to the reference's own
          outputs; OpenMP over trees) with the SAME network evaluated by stock PyTorch CPU kernels, one batched `predict` per
          simulation step exactly as search.py:82-84 does, on all host cores; each step a bounded sample (fewer games) of the
          same workload.  When baseline/_ref holds the reference's own Python (scripts/install_reference.py), its
          `EpisodeGenerator` is timed as well (`reference_python`: BASELINE config 1 exactly, E = 100, and one process per core).
`--dump-outputs DIR`  the episodes the drain after the last timed step returned (rank 0), sorted as `EpisodeGenerator` yields
          them, one float64 DIR/<field>.npy per `EpisodeBatch` field (at most 64 MB: above that, a seeded sample of whole episodes).
          The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark writes nothing there
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NODE_BYTES = 20  # W f64 + N u32 + P f32 + CB u32


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=None, help="total games: default 16384 on one GPU (configs[2]), 65536 sharded over N > 1 (configs[3])")
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--net", default="resnet4x64", help="network in the loop: resnetBxC | basic | cnn")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16", "fp32"], help="operand format of the evaluator (fp32 accumulate)")
    ap.add_argument("--burn-in", type=int, default=36, help="untimed move steps before the warm-up (games reach their stationary mix)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--extras", default="config2,tree_scaling,resnet4x64:fp16,resnet4x64:bf16:pingpong,basic,resnet9x128,cnn",
                    help="side measurements on one GPU, comma separated: config2 | tree_scaling | basic | resnetBxC | cnn | none")
    ap.add_argument("--extra-steps", type=int, default=3)
    ap.add_argument("--cpu-games", type=int, default=256, help="games of the CPU arm's bounded sample")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--trunk-variant", type=int, default=None, help="64-channel ResNet kernel: 4 = filter rows fused, N = 192 (csrc/az_resnet_wide.cu, default), 2 = layer-pipelined, two CTAs per SM (csrc/az_resnet_pipe.cu), 0 = one CTA per SM, 1 = ping-pong (csrc/az_conv.cu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the episodes drained after the last timed step to DIR/<field>.npy (float64) for output comparison between builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def total_games(args, world: int) -> int:
    return args.games if args.games else (16384 if world == 1 else 65536)


def net_label(spec: str) -> str:
    return {"basic": "BasicNN 42-512-512-{7,2}", "cnn": "CNNModel 3-64-128-256 + FC 10752-512"}.get(spec, "ResNet " + spec.replace("resnet", "") + " (blocks x channels)")


def workload_config(args, world: int) -> dict:
    """The workload description both arms print (identical keys and values)."""
    G = total_games(args, world)
    return {"workload": f"connect4_selfplay_{args.net}_{args.dtype}_{G}x{args.sims}", "num_games": G, "num_simulations": args.sims,
            "net": net_label(args.net), "evaluator_dtype": args.dtype, "c_puct": 1.0, "parallelism": f"games sharded x{world}",
            "l2": "no flush: every step streams a tree arena far larger than the 126 MB L2 (2.2 GB at 16384 x 800)"}


def make_model(spec: str, seed: int = 0):
    import torch

    import alphazero_implementation_b200 as az

    torch.manual_seed(seed)
    if spec == "basic":
        return az.BasicNN(), 577_024
    if spec == "cnn":
        return az.CNNModel(), 42_122_000
    b, c = spec.replace("resnet", "").split("x")
    m = az.ResNet(num_res_blocks=int(b), num_channels=int(c))
    return m, m.flops_per_position()


def torch_dtype(name: str):
    import torch

    return {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[name]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))),
                    source="measured (MEASURED_PEAKS.json; bf16 = the sustained figure: the kernel is timed inside a long step)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index: int, period_s: float = 0.1):
        import threading

        self.samples, self.reason_bits, self.power = [], 0, []
        self.stop_flag, self.ok, self.period = False, False, period_s
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")  # NVML enumerates physical GPUs
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as exc:  # pragma: no cover
            self.err = repr(exc)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self) -> dict:
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.t.join(timeout=2)
        sm = sorted(self.samples)
        reasons = sorted(k for k, bit in self.REASONS.items() if self.reason_bits & bit)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "power_w_max": max(self.power) if self.power else None,
                "samples": len(sm), "reasons": reasons, "source": "NVML polled every 100 ms during the timed region"}


def algorithmic_bytes(st: dict) -> int:
    """Bytes the tree kernels must move for the work counted in `st` (DESIGN.md, 'algorithmic bytes')."""
    return (st["children_scanned"] * NODE_BYTES + st["simulations"] * 8 + st["children_created"] * NODE_BYTES
            + st["evaluations"] * 4 + st["backup_nodes"] * 24)


def diff(a: dict, b: dict) -> dict:
    return {k: b[k] - a[k] for k in a}


# --------------------------------------------------------------------------------------------------  CPU arm
def host_cores() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_model_name() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_arm_net(spec: str, E: int, S: int, target_s: float, max_steps: int = 10**6):
    """The reference algorithm on the host cores with the network in the loop: C restatement of the tree search (OpenMP over
    trees) + the same torch module on CPU in fp32, one batched forward per simulation step (search.py:82-84).  A step = one move
    step of E games x S simulations; as many steps as fit in ~target_s (at least one)."""
    import numpy as np
    import torch

    from oracle import c4oracle
    from oracle.net_eval import TorchNetEvaluator

    cores = host_cores()
    cores = c4oracle.set_threads(cores)  # explicit: torchrun exports OMP_NUM_THREADS=1 to its workers
    torch.set_num_threads(cores)
    model, _ = make_model(spec)
    ev = TorchNetEvaluator(model)
    rng = np.random.RandomState(0)
    # probe: a few simulation steps (thread pools, allocator), then size the sample
    t0 = time.perf_counter()
    c4oracle.search(np.zeros(E, np.uint64), np.zeros(E, np.uint64), np.zeros(E, np.uint8), 24, py_eval=ev)
    t_sim = (time.perf_counter() - t0) / 24
    steps = max(1, min(max_steps, int(target_s / max(t_sim * S, 1e-3))))
    t0 = time.perf_counter()
    r = c4oracle.selfplay(E, S, rng.random_sample((steps, E)), quota=10**9, py_eval=ev)
    dt = time.perf_counter() - t0
    return dict(sims_per_s=r.n_sims / dt, games_per_s=len(r.ep_slot) / dt, steps=steps, seconds=dt, cores=cores, ms_per_step=dt / steps * 1e3,
                sims=r.n_sims, evals=r.n_evals, games=E)


def cpu_arm_builtin(E: int, S: int, kind: int, target_s: float = 8.0):
    """Same with a built-in deterministic evaluator (config 2 side measurement)."""
    import numpy as np

    from oracle import c4oracle

    cores = c4oracle.set_threads(host_cores())
    rng = np.random.RandomState(0)
    c4oracle.selfplay(E, S, rng.random_sample((2, E)), quota=10**9, eval_kind=kind)
    t0 = time.perf_counter()
    c4oracle.selfplay(E, S, rng.random_sample((3, E)), quota=10**9, eval_kind=kind)
    t1 = (time.perf_counter() - t0) / 3
    steps = max(1, min(3000, int(target_s / max(t1, 1e-4))))
    t0 = time.perf_counter()
    r = c4oracle.selfplay(E, S, rng.random_sample((steps, E)), quota=10**9, eval_kind=kind)
    dt = time.perf_counter() - t0
    return dict(sims_per_s=r.n_sims / dt, steps=steps, seconds=dt, cores=cores)


def reference_python_leg(budget_s: float = 45.0):
    """The reference's OWN Python (`EpisodeGenerator` -> `AlphaZeroSearch` -> `BasicNN.predict`, imported unchanged from
    baseline/_ref, populated by scripts/install_reference.py) on this host: BASELINE config 1 exactly (scripts/train.py:12-19 with
    E = 1: S = 100, BasicNN, seeds 0, one thread), the reference's production batching E = 100, and one process per core.
    The game under it is the CPU restatement oracle/shims/simulator (the third-party C++ `simulator` 0.0.4 is not available)."""
    import subprocess

    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "alphazero_implementation")):
        return {"unavailable": "baseline/_ref/alphazero_implementation missing (run scripts/install_reference.py where /root/reference exists)"}
    worker = os.path.join(ROOT, "scripts", "time_reference_python.py")
    cores = host_cores()
    out = {"cores": cores, "cpu_model": cpu_model_name(), "game": "oracle/shims/simulator (CPU restatement of simulator 0.0.4)",
           "torch_threads_per_process": 1}

    def run(E, seed, seconds):
        return subprocess.Popen([sys.executable, worker, "--episodes", str(E), "--sims", "100", "--seed", str(seed), "--seconds", str(seconds)],
                                stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1"))

    def collect(procs):
        res = []
        for p in procs:
            so, se = p.communicate(timeout=600)
            if p.returncode != 0:
                raise RuntimeError(se[-500:])
            res.append(json.loads(so.strip().splitlines()[-1]))
        return res

    try:
        per = budget_s / 3
        [c1] = collect([run(1, 0, per)])
        out["config1_E1_S100_basicnn_1core"] = c1
        [e100] = collect([run(100, 0, per)])
        out["E100_S100_basicnn_1process"] = e100
        allc = collect([run(1, s, per) for s in range(cores)])
        out["config1_one_process_per_core"] = {"processes": cores, "sims_per_s": sum(r["sims_per_s"] for r in allc),
                                               "games_per_s": sum(r["games_per_s"] for r in allc)}
    except Exception as exc:  # the port below remains the arm's value
        out["error"] = repr(exc)[:300]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    # K steps of the bounded sample, sized to finish within a few minutes: one probe, then at most K move steps in ~3 x cpu-seconds
    res = cpu_arm_net(args.net, args.cpu_games, args.sims, target_s=max(10.0, 3.0 * args.cpu_seconds), max_steps=max(1, args.steps))
    sample = (f"{res['steps']} move steps of {res['games']} games x {args.sims} sims from the initial position ({res['seconds']:.1f} s): "
              f"oracle/c4_oracle.c (OpenMP over trees) + the same {args.net} torch module in fp32 on {res['cores']} host threads, "
              "one batched forward per simulation step")
    line = {
        "impl": "reference", "metric": "mcts_simulations_per_sec", "value": res["sims_per_s"], "unit": "sims/s", "n_gpus": args.gpus,
        "steps": res["steps"], "warmup": 1, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "games_per_sec": res["games_per_s"],
        "config": workload_config(args, world),
        "cpu_baseline": {"value": res["sims_per_s"], "unit": "sims/s", "cores": res["cores"], "kind": "port", "sample": sample,
                         "cpu_model": cpu_model_name()},
        "e2e": {"value": res["sims_per_s"], "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_python": reference_python_leg(),
        "note": "reference algorithm as the C restatement oracle/c4_oracle.c (pinned to the reference's own outputs), network by stock "
                "PyTorch CPU kernels; `reference_python` = the reference's unmodified Python on this host (its only runnable configs)",
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------  GPU arm
def concat_device(parts: list[dict]) -> dict:
    """Drained episode dicts (device tensors) -> one dict, sample offsets rebased."""
    import torch

    parts = [p for p in parts if p["ep_len"].numel()] or parts[:1]
    out, base = {}, 0
    offs = []
    for p in parts:
        offs.append(p["ep_offset"] + base)
        base += int(p["s_bb0"].numel())
    for k in parts[0]:
        out[k] = torch.cat(offs) if k == "ep_offset" else torch.cat([p[k] for p in parts])
    return out


DUMP_LIMIT_BYTES = 63 << 20  # array bytes: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir: str, drained: dict, limit: int = DUMP_LIMIT_BYTES) -> None:
    """The episodes one drain returned, in the order the public API yields them (move step, then slot), as one float64 .npy per
    `EpisodeBatch` field (bitboards use 49 bits, so float64 holds them exactly).  Above `limit` bytes a fixed seeded sample of
    whole episodes is written instead; the sort comes first, so the sample does not depend on the ring's completion order."""
    import dataclasses

    import numpy as np

    from alphazero_implementation_b200.engine import sort_episode_batch

    b = sort_episode_batch({k: v.cpu().numpy() for k, v in drained.items()})
    cost = 8 * (6 + 10 * b.ep_len.astype(np.int64))  # per episode: slot, step, len, offset, outcome[2]; per sample: bb0, bb1, player, counts[7]
    if cost.sum() > limit:
        order = np.random.RandomState(0).permutation(len(b))
        keep = np.sort(order[np.cumsum(cost[order]) <= limit])
        b = sort_episode_batch(dict(ep_slot=b.ep_slot[keep], ep_step=b.ep_step[keep], ep_len=b.ep_len[keep], ep_offset=b.ep_offset[keep],
                                    ep_outcome=b.ep_outcome[keep], s_bb0=b.s_bb0, s_bb1=b.s_bb1, s_player=b.s_player, s_counts=b.s_counts))
    os.makedirs(out_dir, exist_ok=True)
    for f in dataclasses.fields(b):
        np.save(os.path.join(out_dir, f.name + ".npy"), getattr(b, f.name).astype(np.float64))


def kernel_timing_step(search, eng, u):
    """One more move step, un-graphed, with a CUDA-event pair around every evaluator launch -> list of ms."""
    import torch

    pairs: list = []
    search.simulate(eng, evaluator_events=pairs)
    eng.sample_moves(u)
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in pairs]


def net_extra(args, spec: str, device_index: int, peaks: dict):
    """Side measurement: another network in the loop at 16384 games x S sims on one GPU.  Burn-in with the fused uniform
    evaluator (cheap; a random-init net plays a near-uniform game too), then warm-up + timed move steps with the net."""
    import numpy as np
    import torch

    import alphazero_implementation_b200 as az
    from alphazero_implementation_b200.engine import EVAL_UNIFORM

    spec, dname, variant = (spec.split(":") + ["", ""])[:3]  # "resnet4x64:fp16" = fp16 operands; "resnet4x64:bf16:pingpong" = csrc/az_conv.cu
    dname = dname or ("bf16" if args.dtype == "fp32" else args.dtype)
    model, flops = make_model(spec)
    E, S = 16384, args.sims
    dt = torch_dtype(dname)
    search = az.AlphaZeroSearch(model=model, num_simulations=S, device=device_index, inference_dtype=dt,
                                trunk_variant={"pingpong": 1, "pipe": 0, "pipe2": 2, "pair": 3, "wide": 4}.get(variant))
    eng = search.engine_for(E)
    eng.reset_games()
    n = args.extra_steps
    u = torch.from_numpy(np.random.RandomState(5).random_sample((32 + 2 + n, E))).to(eng.device)
    for i in range(32):
        eng.run_move_step(S, EVAL_UNIFORM, u[i])
        if i % 8 == 7:
            eng.drain_episodes_device()
    search.simulate_and_move(eng, u[32])  # warm-up (graph capture)
    eng.drain_episodes_device()
    torch.cuda.synchronize()
    st0 = eng.stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        search.simulate_and_move(eng, u[33 + i])
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    st = diff(st0, eng.stats())
    k_ms = kernel_timing_step(search, eng, u[33 + n])
    eng.drain_episodes_device()
    k_mean = float(np.mean(k_ms))
    evals_per_launch = st["evaluations"] / (n * S)
    rec = {"workload": f"connect4_selfplay_{spec}_{dname}_{E}x{S}", "net": net_label(spec), "evaluator": search.evaluator_name,
           "move_steps": n, "sims_per_s": st["simulations"] / ms * 1e3, "us_per_sim_step": ms * 1e3 / (n * S),
           "flops_per_position": flops, "evaluator_kernel_us": k_mean * 1e3,
           "tensor_tflops_in_kernel": evals_per_launch * flops / (k_mean * 1e-3) / 1e12,
           "tensor_frac_of_measured_bf16": evals_per_launch * flops / (k_mean * 1e-3) / 1e12 / peaks["bf16_tflops"],
           "leaf_eval_fraction": st["evaluations"] / max(1, st["simulations"])}
    search.close()
    return rec


def config2_extra(args, device_index: int, peaks: dict):
    """BASELINE configs[1] (last round's headline): 4096 games x 200 sims, uniform evaluator, the fused `k_run_sims` move step."""
    import numpy as np
    import torch

    import alphazero_implementation_b200 as az
    from alphazero_implementation_b200.engine import EVAL_UNIFORM

    E, S, K = 4096, 200, 30
    eng = az.Engine(num_games=E, num_simulations=S, device=device_index)
    eng.reset_games()
    u = torch.from_numpy(np.random.RandomState(1000).random_sample((48 + K, E))).to(eng.device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    for i in range(48):
        eng.run_move_step(S, EVAL_UNIFORM, u[i])
        if i % 8 == 7:
            eng.drain_episodes_device()
    torch.cuda.synchronize()
    st0 = eng.stats()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    for i in range(K):
        flush.zero_()
        ev[i][0].record()
        eng.run_move_step(S, EVAL_UNIFORM, u[48 + i])
        ev[i][1].record()
        if i % 8 == 7:
            eng.drain_episodes_device()
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    st = diff(st0, eng.stats())
    gbs = algorithmic_bytes(st) / (ms * 1e-3) / 1e9
    eng.close()
    cpu = cpu_arm_builtin(E, S, 1, target_s=6.0)
    return {"workload": f"connect4_selfplay_uniform_{E}x{S}", "kernel": "k_run_sims (fused search + move, one launch per step)", "steps": K,
            "sims_per_s": st["simulations"] / ms * 1e3, "ms_per_step": ms / K, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peaks["hbm_gbs"],
            "l2": "flushed between steps", "cpu_port_sims_per_s": cpu["sims_per_s"], "cpu_cores": cpu["cores"]}


def tree_scaling(args, device_index: int, peaks: dict):
    """The fused tree kernel (uniform evaluator) at S = 800 and at S = 200 for larger tree counts: latency-bound, so its fraction
    of the HBM roofline grows with the number of independent trees until the issue slots fill."""
    import numpy as np
    import torch

    import alphazero_implementation_b200 as az
    from alphazero_implementation_b200.engine import EVAL_UNIFORM

    out = []
    for E, S in ((4096, 800), (16384, 800), (65536, 800), (16384, 200), (65536, 200)):
        eng = az.Engine(num_games=E, num_simulations=S, device=device_index)
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(5).random_sample((16, E))).to(eng.device)
        for i in range(11):
            eng.run_move_step(S, EVAL_UNIFORM, u[i])
        eng.drain_episodes_device()
        torch.cuda.synchronize()
        st0 = eng.stats()
        ms = 0.0
        for i in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.run_move_step(S, EVAL_UNIFORM, u[11 + i])
            b.record()
            torch.cuda.synchronize()
            ms += a.elapsed_time(b)
        st = diff(st0, eng.stats())
        gbs = algorithmic_bytes(st) / (ms * 1e-3) / 1e9
        out.append({"trees": E, "num_simulations": S, "kernel": "k_run_sims", "kernel_ms": ms / 5, "sims_per_s": st["simulations"] / ms * 1e3,
                    "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peaks["hbm_gbs"], "bytes_per_sim": algorithmic_bytes(st) / max(1, st["simulations"])})
        eng.close()
        del eng
        torch.cuda.empty_cache()
    return out


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import alphazero_implementation_b200 as az

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: everything a library prints there (NCCL's version and communicator lines at the
    # NCCL_DEBUG level the launcher chose, cuDNN notices) is sent to stderr by pointing fd 1 at fd 2; the JSON line goes to the saved fd
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1 and os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
        os.environ["NCCL_DEBUG"] = "INFO"  # communicator lines (rank count per communicator) - on stderr, see above
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from alphazero_implementation_b200.distributed import all_gather_episodes, shard_range

    W, K = max(3, args.warmup), args.steps
    G, S = total_games(args, world), args.sims
    lo, hi = shard_range(G, rank, world)
    E = hi - lo
    peaks = load_peaks()
    model, flops = make_model(args.net)
    # k_resnet_wide's measurement hook: first-CTA start / last-CTA end of every launch on the device's global timer -> the kernel's
    # duration INSIDE the timed region (set before the first launch: the pointer is baked into the captured graph)
    from alphazero_implementation_b200 import _lib as az_lib
    T_CAP = 1 << 15
    timing = torch.zeros(4 + 2 * T_CAP, dtype=torch.int64, device=torch.device("cuda", local))
    timing[4::2] = -1  # ~0 as uint64: atomicMin target
    az_lib.load().az_resnet_wide_set_timing(timing.data_ptr(), T_CAP)
    gen = az.EpisodeGenerator(model=model, num_simulations=S, num_episodes=E, game_initial_state=az.Config(6, 7, 4).sample_initial_state(),
                              device=local, inference_dtype=torch_dtype(args.dtype), trunk_variant=args.trunk_variant)
    search = gen.search
    eng = search.engine_for(E)
    eng.reset_games()
    rng = np.random.RandomState(1000 + rank)
    n_pre = args.burn_in + W
    u_all = torch.from_numpy(rng.random_sample((n_pre + K + 1, E))).to(eng.device)  # inputs resident in HBM

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = []
    for i in range(n_pre):
        search.simulate_and_move(eng, u_all[i])
        d = eng.drain_episodes_device()
        if i >= args.burn_in:
            warm.append(d)
    # the all-gather's slab capacity, known to every rank before the call (one collective, counts in the slab header): games finish at
    # ~E / 20 per step and leave ~1 sample per slot per step; a rank that exceeded it would be seen by all and the exact path taken
    ag_cap = (E * K // 8 + 64, int(1.5 * E * K) + 64 * 42)
    if world > 1:
        all_gather_episodes(concat_device(warm), slot_offset=lo, capacity=ag_cap)  # NCCL channel set-up and buffer sizing belong to the warm-up
    drain_bufs = [eng.alloc_drain_buffers() for _ in range((K + 15) // 16)]  # no allocation inside the timed region
    barrier()
    st0 = eng.stats()
    launch0 = int(timing[0].item())
    timing[4::2] = -1  # fresh slots for the region's launches (at most T_CAP of them)
    timing[5::2] = 0
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    ev0, ev1, ag0 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    t_wall0 = time.perf_counter()
    ev0.record()
    drained = []
    step_ev = [ev0]
    for i in range(K):
        search.simulate_and_move(eng, u_all[n_pre + i])  # 800 x (k_resnet_wide, k_expand_select) replayed from a CUDA graph + k_sample_moves
        if (i + 1) % 16 == 0 or i + 1 == K:  # device -> device; the ring holds 2 E + 64 episodes, ~E / 20 finish per step.  Draining
            drained.append(eng.drain_episodes_device(drain_bufs[i // 16]))  # (a host synchronisation) every step left the GPU queue empty at every
        step_ev.append(torch.cuda.Event(enable_timing=True))  # step boundary: any host hiccup there showed up as a 10 % slower step
        step_ev[-1].record()
    ag0.record()
    merged = concat_device(drained)
    if world > 1:
        merged = all_gather_episodes(merged, slot_offset=lo, capacity=ag_cap)  # configs[3]: every rank ends the region holding every finished episode
    ev1.record()
    barrier()
    wall_s = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launch1 = int(timing[0].item())
    k_region = None
    if 0 < launch1 - launch0 <= T_CAP:
        slots = torch.arange(launch0, launch1, device=timing.device) % T_CAP
        dur = (timing[5::2][slots] - timing[4::2][slots]).double() * 1e-6  # ns -> ms
        k_region = {"launches": launch1 - launch0, "mean_ms": float(dur.mean().item()), "min_ms": float(dur.min().item()), "max_ms": float(dur.max().item())}
    az_lib.load().az_resnet_wide_set_timing(None, 0)  # off for everything that follows (extras build their own graphs)
    st = diff(st0, eng.stats())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, drained[-1])  # the last timed step always drains
    total_ms, ag_ms = ev0.elapsed_time(ev1), ag0.elapsed_time(ev1)
    step_ms = [step_ev[i].elapsed_time(step_ev[i + 1]) for i in range(K)]
    n_eps_job = int(merged["ep_len"].numel())
    if world > 1:
        t = torch.tensor([total_ms, ag_ms], dtype=torch.float64, device=eng.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, ag_ms = float(t[0].item()), float(t[1].item())
        cnt = torch.tensor([st["simulations"], st["evaluations"]], dtype=torch.float64, device=eng.device)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        tot_sims, tot_evals = float(cnt[0].item()), float(cnt[1].item())
    else:
        tot_sims, tot_evals = float(st["simulations"]), float(st["evaluations"])
    value = tot_sims / total_ms * 1e3
    launches = K * search.launches_per_move_step()
    ag_iso_ms = None
    if world > 1:  # the same collective once more from a common start: inside the region its time is mostly the ranks' skew
        local_again = concat_device(drained)
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        all_gather_episodes(local_again, slot_offset=lo, capacity=ag_cap)
        b1.record()
        torch.cuda.synchronize()
        t = torch.tensor([b0.elapsed_time(b1)], dtype=torch.float64, device=eng.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ag_iso_ms = float(t.item())

    # roofline of the dominant kernel on this rank: CUDA events around each evaluator launch of one more (un-graphed) move step
    k_ms = kernel_timing_step(search, eng, u_all[n_pre + K])
    eng.drain_episodes_device()
    k_events = float(np.mean(k_ms))
    # the duration the roofline uses: the kernel's own device-timer stamps inside the timed region (k_resnet_wide), else the events
    # of the extra un-graphed step (between launch gaps the GPU boosts above its power-capped clock: a slight underestimate)
    k_mean = k_region["mean_ms"] if k_region else k_events
    evals_per_launch = st["evaluations"] / (K * S)
    achieved = evals_per_launch * flops / (k_mean * 1e-3) / 1e12
    roofline = {"kernel": search.evaluator_name, "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": achieved / peaks["bf16_tflops"], "traffic": None, "peak_source": peaks["source"],
                "algorithmic_flops_per_launch": evals_per_launch * flops, "flops_per_position": flops, "positions_per_launch": E,
                "evaluated_leaves_per_launch": evals_per_launch, "kernel_ms": k_mean, "kernel_launches_timed": len(k_ms),
                "kernel_ms_events_ungraphed_step": k_events, "kernel_in_timed_region": k_region,
                "kernel_share_of_step": k_mean * S / (ev0.elapsed_time(ev1) / K),
                "how": "k_resnet_wide stamps the device's global timer at its first CTA's start and its last CTA's end (az_resnet_wide_set_timing): "
                       "mean over every launch INSIDE the timed region; other evaluators: CUDA events around each launch of one extra un-graphed "
                       "move step right after the timed region (kernel_ms_events_ungraphed_step, reported for both)",
                # the events of the extra step see the kernel between launch gaps (GPU below its power cap, higher clock); the whole
                # timed step divided by S bounds the in-region duration from above
                "frac_lower_bound_whole_step": evals_per_launch * flops / (ev0.elapsed_time(ev1) / K / S * 1e-3) / 1e12 / peaks["bf16_tflops"],
                "note": "tensor-bound by classification.  k_resnet_wide fuses the three taps of a filter row into one 128x192x16 MMA (96 cycles "
                        "of math; measured 112-115: the A tile is fetched once per 128 output columns, 14 KB of shared-memory operands at 128 "
                        "B/clk) - 12 MMAs per tile-layer instead of 36 of 48 cycles; the epilogue's shuffles / stores share that crossbar, so the "
                        "kernel runs at ~1700 cycles per tile-layer against 1152 of math (ncu: tensor pipe 65.9 %, profiles/"
                        "r02_k_resnet_wide_steady_ncu_raw.json); the previous 64-channel kernel (k_resnet_pipe, N = 64) measured 0.47",
                "tree_kernel": {"name": "k_expand_select", "us_per_launch": (ev0.elapsed_time(ev1) / K / S - k_mean) * 1e3,
                                "algorithmic_gbs": algorithmic_bytes(st) / K / S / max(1e-9, (ev0.elapsed_time(ev1) / K / S - k_mean) * 1e-3) / 1e9,
                                "note": "step time minus evaluator time; latency-bound pointer chasing, see DESIGN.md"}}
    prof = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(prof):
        try:
            roofline["traffic"] = json.load(open(prof)).get(search.evaluator_name + "_dram_bytes_per_launch")
        except Exception:
            pass

    # end to end through the public API with host buffers, continuing the same games
    e2e = None
    if not args.no_e2e:
        np.random.seed(7 + rank)
        W2 = 2
        batches, e2e_t0, sims_before, bytes0 = [], None, None, (0, 0)
        for step, batch, _ in gen.iter_steps(max_steps=W2 + K + 1, reset=False):
            if step == W2 - 1:  # warm-up done: open the timed region on a quiet device (step W2 is already enqueued: it is
                barrier()       # finished by this barrier and counted as warm-up by the statistics snapshot below)
                sims_before = eng.stats()
                bytes0 = (gen.h2d_bytes, gen.d2h_bytes)
                e2e_t0 = time.perf_counter()
                continue
            if e2e_t0 is not None and batch is not None:
                batches.append(batch)
        n_eps = sum(len(b) for b in batches)
        if world > 1:
            from alphazero_implementation_b200.trainer import _concat, _to_device

            loc = batches[0]
            for b in batches[1:]:
                loc = _concat(loc, b)
            n_eps = int(all_gather_episodes(_to_device(loc, eng.device), slot_offset=lo)["ep_len"].numel())
        barrier()
        e2e_s = time.perf_counter() - e2e_t0
        d = diff(sims_before, eng.stats())
        n_steps = d["moves"] // E
        h2d, d2h = gen.h2d_bytes - bytes0[0], gen.d2h_bytes - bytes0[1]
        t = torch.tensor([e2e_s], dtype=torch.float64, device=eng.device)
        c = torch.tensor([float(d["simulations"])], dtype=torch.float64, device=eng.device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
        e2e = {"value": float(c.item()) / float(t.item()), "unit": "sims/s", "h2d_bytes_per_step": int(h2d / max(1, n_steps)),
               "d2h_bytes_per_step": int(d2h / max(1, n_steps)), "steps": int(n_steps), "games_per_sec": n_eps / float(t.item()),
               "api": "EpisodeGenerator.iter_steps: pinned-host uniforms in, finished episodes + ring counters out to pinned host memory every "
                      "step (readback of step k overlaps step k+1)" + ("; then the NCCL all-gather of the region's episodes" if world > 1 else "")}

    arena_bytes = eng.device_bytes
    details = {"games_per_gpu": E, "burn_in_steps": args.burn_in, "tree_arena_bytes": arena_bytes, "evaluator": search.evaluator_name,
               "flops_per_position": flops, "leaf_eval_fraction": tot_evals / max(1.0, tot_sims),
               "us_per_simulation_step": total_ms * 1e3 / (K * S), "cuda_graph": bool(search.use_cuda_graph),
               "episodes_finished_in_timed_region": n_eps_job, "step_ms": [round(x, 2) for x in step_ms]}
    dev_file = os.path.join(ROOT, "profiles", "r02_evaluator_deviation.json")  # written by tests/test_gpu_config3.py on 16384 positions
    if os.path.exists(dev_file):
        try:
            dev = json.load(open(dev_file))
            details["evaluator_max_abs_dev_vs_fp32_predict"] = {k: dev[k] for k in (f"{args.net}_{args.dtype}", f"{args.net}_fp16") if k in dev}
        except Exception:
            pass
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_arm_net(args.net, args.cpu_games, S, target_s=args.cpu_seconds)
            cpu = {"value": r["sims_per_s"], "unit": "sims/s", "cores": r["cores"], "kind": "port", "cpu_model": cpu_model_name(),
                   "sample": f"{r['steps']} move steps of {r['games']} games x {S} sims from the initial position ({r['seconds']:.1f} s): oracle/c4_oracle.c with "
                             f"OpenMP over trees + the same {args.net} torch module in fp32 on the host cores, one batched forward per simulation step"}
        except Exception as exc:
            cpu = {"error": repr(exc)[:300]}
    search.close()
    del gen, search, eng
    torch.cuda.empty_cache()

    extras = {}
    if rank == 0 and world == 1:
        for spec in [s for s in args.extras.split(",") if s and s != "none"]:
            try:  # side measurements must not sink the headline
                if spec == "config2":
                    extras["config2"] = config2_extra(args, local, peaks)
                elif spec == "tree_scaling":
                    extras["tree_scaling"] = tree_scaling(args, local, peaks)
                elif spec != args.net + ":" + args.dtype and spec != args.net:
                    extras.setdefault("net_in_loop", []).append(net_extra(args, spec, local, peaks))
            except Exception as exc:
                extras.setdefault("errors", {})[spec] = repr(exc)[:300]
            torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": "mcts_simulations_per_sec", "value": value, "unit": "sims/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic", "games_per_sec": n_eps_job / total_ms * 1e3, "config": workload_config(args, world), "details": details,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "wall_s_timed_region": wall_s, "work_per_step": {k: v / K for k, v in st.items()},
        }
        if world > 1:
            line["episode_allgather"] = {"ms_in_region_incl_rank_skew": ag_ms, "ms_isolated": ag_iso_ms, "inside_timed_region": True, "collectives": 1,
                                         "episodes": n_eps_job, "samples": int(merged["s_bb0"].numel()), "slab_capacity": list(ag_cap)}
        line.update(extras)
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
