#!/usr/bin/env python
"""Cost of the action masks (td_action_mask) at the batch sizes of bench.py's workloads.

    python tools/mask_bench.py [--steps K] [--repeats R] [--out FILE]

Per workload, CUDA events around K launches, R repeats, median of the repeats:
  step       TDVecEnv.step alone, ms per step
  step+mask  step followed by action_mask(), ms per step
  mask       action_mask() alone on the state the steps left, ms per launch; the bytes it reads (about 300 per env on
             10x10 boards) fit in L2, so repeated launches read them from there, not from HBM
and the mask kernel's algorithmic bytes (header, map6 + MapHdr, the live towers read; n (6 L^2 + 1) and n 12 bytes
written) over its time, against the 6534.8 GB/s copy peak of DESIGN.md.  The card's name and power limit are printed
with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

COPY_PEAK_GBS = 6534.8
# (kind, L, envs, multi): the batch sizes of bench.py's workloads def-small, def-middle-multi, atk-small, 2p-large
WORKLOADS = {"def-small": ("def", 10, 65536, False), "def-middle-multi": ("def", 20, 32768, True),
             "atk-small": ("atk", 10, 65536, False), "2p-large": ("2p", 30, 16384, False)}


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power or "unknown"


def timed(torch, fn, k, repeats):
    runs = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(k):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        runs.append(a.elapsed_time(b) / k)
    return statistics.median(runs), runs


def mask_bytes(env):
    """Bytes the mask kernel reads and writes for the current state of `env`."""
    from gym_td_b200 import engine as E
    import numpy as np
    n, L = env.num_envs, env.map_size
    cells_pad = (L * L + 15) & ~15
    hdr = env.engine.get_state_raw()[:, :64].copy().view(E.HEADER_DTYPE).reshape(-1)
    read = 64 * n
    written = 0
    if env.kind != "atk":
        read += n * (cells_pad + 16) + 16 * int(np.sum(hdr["n_towers"], dtype=np.int64))
        written += n * (6 * L * L + 1)
    else:
        read += 16 * n                                       # the MapHdr alone
    if env.kind != "def":
        written += 12 * n
    return read, written


def run(name, steps, repeats, warmup):
    import torch
    from gym_td_b200.vec_env import TDVecEnv
    kind, L, n, multi = WORKLOADS[name]
    dev = torch.device("cuda", 0)
    env = TDVecEnv(kind, L, n, seed=0, auto_reset=True, multi_action=multi)
    env.reset()
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    pool = 8
    if multi:
        d = (torch.rand((pool, n, 6, L, L), device=dev, generator=g) < 0.01).to(torch.int64)
    else:
        d = torch.randint(0, 6 * L * L + 1, (pool, n), dtype=torch.int64, device=dev, generator=g)
    a = torch.randint(0, 5, (pool, n, 3, 8), dtype=torch.int64, device=dev, generator=g)
    act = [{"def": d[k], "atk": a[k], "2p": {"Attacker": a[k], "Defender": d[k]}}[kind] for k in range(pool)]
    for i in range(warmup):
        env.step(act[i % pool])
        if i % 4 == 0:
            env.action_mask()
    torch.cuda.synchronize()
    step_ms, step_runs = timed(torch, lambda i: env.step(act[i % pool]), steps, repeats)
    both_ms, both_runs = timed(torch, lambda i: (env.step(act[i % pool]), env.action_mask()), steps, repeats)
    mask_ms, mask_runs = timed(torch, lambda i: env.action_mask(), steps, repeats)
    read, written = mask_bytes(env)
    gbs = (read + written) / (mask_ms * 1e-3) / 1e9
    env.close()
    return {"workload": name, "kind": kind, "L": L, "envs": n, "multi_action": multi, "steps_per_repeat": steps,
            "repeats": repeats, "step_ms": step_ms, "step_plus_mask_ms": both_ms, "mask_added_ms": both_ms - step_ms,
            "mask_ms": mask_ms, "mask_bytes_read": read, "mask_bytes_written": written, "mask_GBs": gbs,
            "mask_fraction_of_copy_peak": gbs / COPY_PEAK_GBS,
            "runs_ms": {"step": step_runs, "step_plus_mask": both_runs, "mask": mask_runs}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="launches per timed repeat")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--workload", action="append", choices=sorted(WORKLOADS))
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mask_bench.py needs a CUDA device; nothing is measured on the CPU")
    name, power = card()
    lines = [json.dumps({"card": name, "power_limit": power})]
    print(lines[0], flush=True)
    for w in args.workload or list(WORKLOADS):
        r = run(w, args.steps, args.repeats, args.warmup)
        r.update(card=name, power_limit=power)
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
