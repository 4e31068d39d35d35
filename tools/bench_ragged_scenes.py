"""Scenes of different sizes: one ragged SirenTrainer (n_coords = a list of counts) against T single-scene captured
trainers stepped back to back and, where every scene has the same count, the equal-N T-scene trainer.

Cases (bf16, 3 x 256 hidden, in 2 / out 1, image_mse, no clip):
  mix   16 scenes drawn (seeded) from 64^2, 128^2, 256^2 and 512^2 coordinates
  eq64  64 scenes of 4,096 coordinates given as a list (the equal-N trainer runs the same units)
The arms are timed alternately in one process (CUDA events around `--rounds` rounds; a round is one step of all T
scenes).  Reported per arm: ms per round (median of the `--reps` alternations, and the spread), Mcoord/s, and the
per-kernel breakdown of one round (siren_b200_profile_begin/end around non-graph steps, a separate pass).  The GPU name
and power limit are read in the same run.

    python tools/bench_ragged_scenes.py [--cases mix,eq64] [--rounds 20] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import random
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_multi_scene import gpu_info, profile_round, time_rounds  # noqa: E402
from siren_mri_b200 import modules  # noqa: E402
from siren_mri_b200.trainer import SirenTrainer  # noqa: E402


def counts_of(case):
    if case == "mix":
        rng = random.Random(0)
        return [rng.choice([64 * 64, 128 * 128, 256 * 256, 512 * 512]) for _ in range(16)]
    if case == "eq64":
        return [4096] * 64
    raise SystemExit("unknown case %r" % case)


def make_arms(counts, seed=0):
    torch.manual_seed(seed)
    T = len(counts)
    net = lambda: modules.SingleBVPNet(in_features=2, out_features=1, precision="bf16").cuda()  # noqa: E731
    models = [net() for _ in range(T)]
    states = [m.net.state_dict() for m in models]
    total = sum(counts)
    coords = torch.rand(total, 2, device="cuda") * 2 - 1
    gt = torch.rand(total, 1, device="cuda") * 2 - 1
    arms = {}
    ragged = SirenTrainer(models, list(counts), lr=1e-4)
    ragged.coords.copy_(coords)
    ragged.gt.copy_(gt)
    arms["ragged"] = ragged
    singles, x0 = [], 0
    for t, n in enumerate(counts):
        s = SirenTrainer(net(), n, lr=1e-4)
        s.block.load_state_dict(states[t])
        s.refresh_weights()
        s.coords.copy_(coords[x0:x0 + n].view(1, n, 2))
        s.gt.copy_(gt[x0:x0 + n].view(1, n, 1))
        x0 += n
        singles.append(s)
    arms["singles"] = singles
    if len(set(counts)) == 1:
        eq_models = [net() for _ in range(T)]
        for m, st in zip(eq_models, states):
            m.net.load_state_dict(st)
        eq = SirenTrainer(eq_models, counts[0], lr=1e-4)
        eq.coords.copy_(coords.view(T, counts[0], 2))
        eq.gt.copy_(gt.view(T, counts[0], 1))
        eq.refresh_weights()
        arms["equal_n"] = eq
    return arms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="mix,eq64")
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged_scenes needs a CUDA device")
    name, power = gpu_info()
    result = dict(gpu=name, power_limit_and_max_sm_clock=power, rounds=args.rounds, reps=args.reps, cases=[])
    print("# %s, power limit / max SM clock: %s" % (name, power))
    for case in args.cases.split(","):
        counts = counts_of(case)
        arms = make_arms(counts)
        trainers = {k: (v if isinstance(v, list) else [v]) for k, v in arms.items()}
        steps = {k: (lambda ts=ts: [t.step() for t in ts]) for k, ts in trainers.items()}
        for step in steps.values():
            for _ in range(args.warmup):
                step()
        torch.cuda.synchronize()
        times = {k: [] for k in steps}
        for _ in range(args.reps):      # alternate the arms
            for k, step in steps.items():
                times[k].append(time_rounds(step, args.rounds))
        total = sum(counts)
        row = dict(case=case, T=len(counts), counts=sorted(set(counts)), coords=total)
        for k, ts in times.items():
            med = sorted(ts)[len(ts) // 2]
            row[k] = dict(ms_per_round=round(med, 4), ms_min=round(min(ts), 4), ms_max=round(max(ts), 4),
                          mcoord_per_s=round(total / med / 1e3, 1), kernels=profile_round(trainers[k]))
        for k in steps:
            if k != "ragged":
                row["speedup_vs_" + k] = round(row[k]["ms_per_round"] / row["ragged"]["ms_per_round"], 3)
        result["cases"].append(row)
        print("%s T=%d coords=%d  " % (case, len(counts), total) + "  ".join(
            "%s %.3f ms/round (%.0f Mcoord/s)" % (k, row[k]["ms_per_round"], row[k]["mcoord_per_s"]) for k in steps))
        for k in steps:
            print("  %-8s %s" % (k, "  ".join("%s %.3f ms/%d" % (kn, v["ms"], v["launches"])
                                             for kn, v in row[k]["kernels"].items())))
        del arms, trainers, steps
        torch.cuda.empty_cache()
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
