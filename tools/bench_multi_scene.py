"""Many small scenes: one T-scene SirenTrainer against T single-scene captured trainers stepped back to back.

For each (T, N) the two arms train the same T scenes of N coordinates (bf16, 3 x 256 hidden, image_mse, no clip) and
are timed alternately in one process (CUDA events around `--rounds` rounds; a round is one step of all T scenes).
Reported per arm: ms per round (median of the `--reps` alternations, and the spread), Mcoord/s, and the per-kernel
breakdown of one round (siren_b200_profile_begin/end around non-graph steps, a separate pass: the event brackets slow
the host).  The GPU name and power limit are read in the same run.

    python tools/bench_multi_scene.py [--cases 64x4096,64x16384,16x65536] [--rounds 20] [--reps 3] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from siren_mri_b200 import _lib, modules  # noqa: E402
from siren_mri_b200.trainer import SirenTrainer  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def make_arms(T, n, seed=0):
    torch.manual_seed(seed)
    models = [modules.SingleBVPNet(in_features=2, out_features=1, precision="bf16").cuda() for _ in range(T)]
    coords = torch.rand(T, n, 2, device="cuda") * 2 - 1
    gt = torch.rand(T, n, 1, device="cuda") * 2 - 1
    singles = []
    for t, m in enumerate(models):
        s = SirenTrainer(modules.SingleBVPNet(in_features=2, out_features=1, precision="bf16").cuda(), n, lr=1e-4)
        s.block.load_state_dict(m.net.state_dict())
        s.refresh_weights()
        s.coords.copy_(coords[t:t + 1])
        s.gt.copy_(gt[t:t + 1])
        singles.append(s)
    multi = SirenTrainer(models, n, lr=1e-4)
    multi.coords.copy_(coords)
    multi.gt.copy_(gt)
    return multi, singles


def time_rounds(step, rounds):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(rounds):
        step()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / rounds


def profile_round(trainers):
    """Per-kernel ms of one round, through the library's event brackets (non-graph steps)."""
    lib = _lib.load()
    for tr in trainers:
        tr.use_graph = False
    torch.cuda.synchronize()
    lib.siren_b200_profile_begin()
    for tr in trainers:
        tr.step()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    _lib.check(lib.siren_b200_profile_end(buf, len(buf)), "profile_end")
    for tr in trainers:
        tr.use_graph = True
    out = {}
    for ln in buf.value.decode().strip().splitlines():
        name, count, ms = ln.split()
        out[name] = dict(launches=int(count), ms=round(float(ms), 4))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="64x4096,64x16384,16x65536")
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multi_scene needs a CUDA device")
    name, power = gpu_info()
    result = dict(gpu=name, power_limit_and_max_sm_clock=power, rounds=args.rounds, reps=args.reps, cases=[])
    print("# %s, power limit / max SM clock: %s" % (name, power))
    for case in args.cases.split(","):
        T, n = (int(v) for v in case.split("x"))
        multi, singles = make_arms(T, n)
        arms = {"multi": multi.step, "singles": lambda: [s.step() for s in singles]}
        for step in arms.values():
            for _ in range(args.warmup):
                step()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for _ in range(args.reps):      # alternate the arms
            for k, step in arms.items():
                times[k].append(time_rounds(step, args.rounds))
        row = dict(T=T, N=n)
        for k, ts in times.items():
            med = sorted(ts)[len(ts) // 2]
            row[k] = dict(ms_per_round=round(med, 4), ms_min=round(min(ts), 4), ms_max=round(max(ts), 4),
                          mcoord_per_s=round(T * n / med / 1e3, 1))
        row["multi"]["kernels"] = profile_round([multi])
        row["singles"]["kernels"] = profile_round(singles)
        row["speedup"] = round(row["singles"]["ms_per_round"] / row["multi"]["ms_per_round"], 2)
        result["cases"].append(row)
        print("T=%d N=%d  multi %.3f ms/round (%.0f Mcoord/s)  singles %.3f ms/round (%.0f Mcoord/s)  x%.2f"
              % (T, n, row["multi"]["ms_per_round"], row["multi"]["mcoord_per_s"], row["singles"]["ms_per_round"],
                 row["singles"]["mcoord_per_s"], row["speedup"]))
        for k in ("multi", "singles"):
            print("  %-8s %s" % (k, "  ".join("%s %.3f ms/%d" % (kn, v["ms"], v["launches"])
                                             for kn, v in row[k]["kernels"].items())))
        del multi, singles, arms
        torch.cuda.empty_cache()
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
