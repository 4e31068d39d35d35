#!/usr/bin/env python
"""bench.py -- SIREN train-step throughput (coords/sec, fwd + bwd + Adam) on N B200s.

Headline workload (BASELINE.json configs[1], "cfg2"): SIREN 3x256, in = 2, out = 1, full-batch 512x512 =
262,144 coordinates per step, synthetic image, MSE (loss_functions.image_mse, high_freq=False), Adam.
A "step" = one pass of the hot path over that batch: forward (which also forms the loss and its gradient), input-
gradient chain, weight gradients, gradient all-reduce (N > 1) and the fused Adam update: four kernel launches of this
library, replayed as one CUDA graph.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision bf16|fp32] [--scaling weak|strong] [--quick]
                  [--dump-outputs DIR]
  python bench.py --impl reference ...    # the reference's own CPU path on the host cores

Prints ONE JSON line (rank 0).  Multi-GPU: launched by torch.distributed.run, one rank per GPU.

Keys of the line beyond the driver's contract (all measured in this run, N = 1 unless noted):
  sustained          the same step timed over >= 2 s (the K-step region is ~0.1 s at boost clocks)
  parity_mode        cfg2 in the fp32-parity mode (bf16 x 3 operand split, rel err <= 1e-4): the mode the north star's
                     tolerance is stated for
  mri_blocks         Fourier blocks of the MRI script (F = 30, 128; in_features 60, 256) at 8 tasks x 65,536 coordinates,
                     bf16 mode, forward + MSE + backward: features built inside the kernels vs materialised every step
  mri_step           one GPU's share of the neural-process step around the hypo-network (8 slices x 65,536 coordinates:
                     hypernetwork -> per-slice SIREN on Fourier features -> k-space data consistency -> image / latent /
                     hypo-weight losses -> backward into the hypernetwork; the encoder is skipped via 'embedding'):
                     native (features, data consistency and weight operands fused into the kernels), the same as ONE
                     CUDA graph, native without those fusions, the reference classes in eager PyTorch
  configs            cfg1..cfg5 through the PUBLIC module API (model -> reference loss -> backward -> torch Adam), native
                     bf16 / native fp32-parity / the reference's ops in eager PyTorch on the same GPU
  gpu_eager_baseline cfg2 with the reference's ops in eager PyTorch on this GPU (fp32, TF32 off) and the ratio to it
  strong             (N > 1) cfg2's ONE 262,144-coordinate batch sharded over the N GPUs, next to the weak value, with
                     the speed-up over one GPU running the whole batch in the same job
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SIDE = 512
N_COORDS = SIDE * SIDE
D_IN, D_OUT, HIDDEN, N_HIDDEN = 2, 1, 256, 3
U = 2 * (D_IN * HIDDEN + N_HIDDEN * HIDDEN * HIDDEN + HIDDEN * D_OUT)      # forward FLOP / coordinate
FLOP_PER_COORD = 3 * U                                                      # fwd + dgrad + wgrad (SURVEY 8d)
HIDDEN_LAYER_FLOP = 2 * HIDDEN * HIDDEN                                     # one 256x256 layer, per coordinate
METRIC = "siren_train_step_coords_per_sec"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained"),
                "hbm_gbs": p["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


def config_dict(world, scaling):
    """The workload both arms (native and --impl reference) are measured on: identical in the two JSON lines."""
    n_local = N_COORDS if scaling == "weak" else (N_COORDS + world - 1) // world
    n_global = N_COORDS * world if scaling == "weak" else N_COORDS
    return {"workload": "cfg2: SIREN 3x256 image fit, 512x512 = 262144 coords/step%s, MSE + Adam"
                        % (" per GPU" if scaling == "weak" and world > 1 else ""),
            "coords_per_step_global": n_global, "coords_per_gpu": n_local, "parallelism": "coords-dp%d" % world,
            "flop_per_coord": FLOP_PER_COORD,
            "l2": "inputs larger than L2: a step streams ~1.9 GB of stash / adjoint planes through the 126 MB L2"}


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (NVML, ~2 ms per sample; falls back to
    polling nvidia-smi when the NVML binding is unavailable)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], False, None
        self.nvml, self.handle = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES-style remapping when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                parts = [v.strip() for v in vis.split(",")]
                if index < len(parts) and parts[index].isdigit():
                    phys = int(parts[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        flags = [bool(r & n.nvmlClocksEventReasonHwSlowdown), bool(r & n.nvmlClocksEventReasonHwThermalSlowdown),
                 bool(r & n.nvmlClocksEventReasonSwThermalSlowdown), bool(r & n.nvmlClocksEventReasonSwPowerCap)]
        self.samples.append((sm, mx, flags))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
        parts = [p.strip() for p in out.stdout.strip().split(",")]
        if len(parts) >= 6 and parts[0].isdigit() and parts[1].isdigit():
            self.samples.append((int(parts[0]), int(parts[1]), [p.lower().startswith("active") for p in parts[2:6]]))

    def _run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=10)
        sm = sorted(s[0] for s in self.samples)
        mx = [s[1] for s in self.samples]
        reasons = sorted({self.NAMES[i] for s in self.samples for i in range(4) if s[2][i]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------------------------
# the reference's own CPU implementation of the path (bench.py --impl reference, and the cpu_baseline leg)
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_seconds(n_coords, steps, warmup, threads):
    """Seconds per training step of the reference on the host cores: (seconds, kind, what).

    kind 'reference': the UNMODIFIED reference classes staged in baseline/_ref (modules.SingleBVPNet ->
    loss_functions.image_mse(high_freq=False) -> backward -> torch.optim.Adam.step, the loop body of
    training.py:66-103); kind 'port': oracle/siren_ref_port.py, the torch-CPU restatement of the same ops, when the
    reference files are not staged on this box."""
    import torch
    torch.set_num_threads(threads)
    from tools import workloads
    ref = workloads.reference_modules()
    if ref is None:
        from oracle import siren_ref_port
        return (siren_ref_port.time_steps(n_coords, steps=steps, warmup=warmup, threads=threads), "port",
                "oracle/siren_ref_port.py (torch CPU ops restating modules.py:25-26,38 + autograd + Adam)")
    torch.manual_seed(0)
    model = workloads.reference_model(D_IN, D_OUT)
    optim = torch.optim.Adam(lr=1e-4, params=model.parameters())
    g = torch.Generator().manual_seed(0)
    coords = torch.rand((1, n_coords, D_IN), generator=g) * 2 - 1
    gt = {"img": torch.rand((1, n_coords, D_OUT), generator=g) * 2 - 1}

    def step():
        out = model({"coords": coords})
        loss = ref[1].image_mse(None, out, gt, high_freq=False)["img_loss"]
        optim.zero_grad()
        loss.backward()
        optim.step()
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return ((time.perf_counter() - t0) / max(steps, 1), "reference",
            "unmodified reference staged in baseline/_ref: modules.SingleBVPNet + loss_functions.image_mse + "
            "torch.optim.Adam on CPU")


def run_reference(args, emit):
    """The reference's CPU implementation of the path, all host threads, bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    import torch
    threads = os.cpu_count() or 1
    # bounded sample: one probe step at full size; if K + W full steps would not end within a few
    # minutes, every step processes a proportionally smaller slice of the 262144 coordinates
    probe, kind, what = cpu_reference_seconds(N_COORDS, 1, 0, threads)
    budget_s = 150.0
    total = (args.steps + max(args.warmup, 1)) * probe
    sample_n = N_COORDS
    if total > budget_s:
        sample_n = max(8192, int(N_COORDS * budget_s / total) // 1024 * 1024)
    sec, kind, what = cpu_reference_seconds(sample_n, args.steps, max(args.warmup, 1), threads)
    value = sample_n / sec
    sample_txt = ("full 262144-coord step" if sample_n == N_COORDS else
                  "%d-coord slice of the 262144-coord step (bounded run time)" % sample_n)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "coords/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_dict(world, args.scaling),
        "mode": {"device": "cpu", "coords_per_timed_step": sample_n},
        "cpu_baseline": {"value": value, "unit": "coords/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": "%s x %d; %s" % (sample_txt, args.steps, what)},
        "e2e": {"value": value, "unit": "coords/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ----------------------------------------------------------------------------------------------------------------
# the native arm
# ----------------------------------------------------------------------------------------------------------------
def synthetic_batch(n_local, rank, world, scaling):
    """A 512x512 grid in [-1,1]^2 (per rank: its shard; under weak scaling its 512 columns of a 512 x (512 world)
    strip) and a smooth synthetic image in [-1,1] -- ONE function of the coordinates, the same on every rank."""
    import torch
    from tools import workloads
    lin = torch.linspace(-1, 1, SIDE)
    lin_x = lin
    if scaling == "weak" and world > 1:
        lin_x = torch.linspace(-1.0 + 2.0 * rank / world, -1.0 + 2.0 * (rank + 1) / world, SIDE + 1)[:-1]
    grid = torch.stack(torch.meshgrid(lin, lin_x, indexing="ij"), dim=-1).reshape(-1, 2)
    if n_local != N_COORDS:
        from siren_mri_b200.parallel import shard_bounds
        b, e = shard_bounds(N_COORDS, rank, world)
        grid = grid[b:e]
        if grid.shape[0] < n_local:
            grid = torch.cat([grid, grid[:n_local - grid.shape[0]]], dim=0)
    img = workloads.synthetic_image(grid)
    return grid.unsqueeze(0).contiguous().pin_memory(), img.unsqueeze(0).contiguous().pin_memory()


def timed_steps(trainer, steps, barrier, dev, world):
    """ms per step over ``steps`` replays: CUDA events, barrier + synchronize on both sides, max over ranks."""
    import torch
    import torch.distributed as dist
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        trainer.step()
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps


def dump_outputs(out_dir, trainer, model):
    """What the last step gave its caller, as float32 ``out_dir/<name>.npy``: the loss, the model output on this
    rank's coordinates (``model_out``, [1, N, 1]) and every parameter after the Adam update (by its state_dict name).
    The loss and model_out come from that step's forward, before its update, so model_out is not model(parameters).
    About 2 MB for cfg2; the inputs are fixed by the arguments, so two builds can be compared output for output.
    Not bit for bit: the weight gradients and the loss are summed with atomic adds, so two runs of one build differ by
    rounding (relative L2 ~1e-4 in model_out after 5 + 50 bf16 steps, measured on one B200 at 1000 W)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": trainer.loss, "model_out": trainer.y}
    arrays.update((name, p) for name, p in model.named_parameters())
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def main():
    # the contract is ONE JSON line on stdout: keep everything libraries print there (NCCL's version banner, ...) on
    # stderr and write the line to the real stdout at the end
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline numbers only (no config table / parity / eager legs)")
    ap.add_argument("--comm", default="auto", choices=["auto", "p2p", "c_abi"],
                    help="N > 1: gradient all-reduce fused into the Adam kernel over peer memory (p2p; auto falls back "
                         "to NCCL when symmetric memory is unavailable) or one ncclAllReduce per step (c_abi)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native step only")
    if args.impl == "reference":
        args.steps = 5 if args.steps is None else args.steps
        args.warmup = 1 if args.warmup is None else args.warmup
        return run_reference(args, emit)
    args.steps = 200 if args.steps is None else args.steps
    args.warmup = 10 if args.warmup is None else max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from siren_mri_b200 import _lib, modules
    from siren_mri_b200.trainer import SirenTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.siren_b200_device_ok(), "siren_b200_device_ok")
    pk = peaks()

    cfg = config_dict(world, args.scaling)
    n_local, n_global = cfg["coords_per_gpu"], cfg["coords_per_step_global"]

    def make_trainer(n, precision, use_dist=True):
        torch.manual_seed(0)
        model = modules.SingleBVPNet(in_features=D_IN, out_features=D_OUT, hidden_features=HIDDEN,
                                     num_hidden_layers=N_HIDDEN, precision=precision).to(dev)
        if world > 1:
            for p in model.parameters():
                dist.broadcast(p.data, 0)
        tr = SirenTrainer(model, n, lr=1e-4, loss_weight=1.0 / 16384.0, precision=precision,
                          use_graph=not args.no_graph, distributed=use_dist, comm=args.comm)
        return model, tr

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def log(msg):
        if rank == 0:
            print("[bench] %s" % msg, file=sys.stderr, flush=True)

    model, trainer = make_trainer(n_local, args.precision)
    comm_used = None if world == 1 else ("fused into the Adam kernel over NVLink peer memory (symmetric memory)"
                                         if trainer.p2p is not None else "ncclAllReduce in the step's graph")
    coords_host, gt_host = synthetic_batch(n_local, rank, world, args.scaling)
    trainer.coords.copy_(coords_host)
    trainer.gt.copy_(gt_host)

    # ---------------- device-resident timing: W warm-up, K timed steps ----------------
    log("warm-up (world=%d, n_local=%d)" % (world, n_local))
    for _ in range(args.warmup):
        trainer.step()
    barrier()
    log("timed region")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_step = timed_steps(trainer, args.steps, barrier, dev, world)
    clocks = sampler.stop() if sampler else None
    value = n_global / (ms_step * 1e-3)
    loss_after = float(trainer.loss.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, model)

    # the same step over >= 2 s: the K-step region above is ~0.1 s at boost clocks
    sustained = None
    if not args.quick:
        log("sustained (>= 2 s)")
        k_sus = max(args.steps, int(2.2 / (ms_step * 1e-3)))
        sampler2 = ClockSampler(local_rank) if rank == 0 else None
        if sampler2:
            sampler2.start()
        ms_sus = timed_steps(trainer, k_sus, barrier, dev, world)
        ck2 = sampler2.stop() if sampler2 else None
        v_sus = n_global / (ms_sus * 1e-3)
        sustained = {"steps": k_sus, "seconds": ms_sus * k_sus * 1e-3, "ms_per_step": ms_sus,
                     "value": v_sus, "unit": "coords/s",
                     "step_frac_of_peak": FLOP_PER_COORD * v_sus / world / 1e12 / pk["bf16_tflops"],
                     "step_frac_of_sustained_peak": (FLOP_PER_COORD * v_sus / world / 1e12 /
                                                     pk["bf16_tflops_sustained"]) if pk["bf16_tflops_sustained"] else None,
                     "clocks": ck2}

    # ---------------- end-to-end through the public API with host buffers ----------------
    log("end-to-end")
    # every step uploads its batch (pinned host memory -> device) and its loss is read back on the host, all inside
    # the timed region; the public call is the pipelined one: the loss of step k is read after step k+1 has been
    # submitted, so the upload of k+1 runs under the kernels of k (SirenTrainer.submit_from_host)
    e2e_steps = max(5, min(args.steps, 100))
    for _ in range(8):
        trainer.submit_from_host(coords_host, gt_host).result()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    prev, e2e_loss = None, None
    for _ in range(e2e_steps):
        h = trainer.submit_from_host(coords_host, gt_host)
        if prev is not None:
            e2e_loss = prev.result()
        prev = h
    e2e_loss = prev.result()
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item()) / e2e_steps
    e2e = {"value": n_global / (e2e_ms * 1e-3), "unit": "coords/s",
           "h2d_bytes_per_step": int(coords_host.numel() * 4 + gt_host.numel() * 4) * world,
           "d2h_bytes_per_step": 4 * world, "ms_per_step": e2e_ms,
           "api": "SirenTrainer.submit_from_host (loss read one step late)", "last_loss": e2e_loss}

    # ---------------- per-kernel timing (CUDA events around each launch, ungraphed) ----------------
    # every rank runs the same steps (they contain the gradient all-reduce); rank 0 records events
    roofline, kernel_table = None, None
    launches_per_step = trainer.kernels_per_step          # replaced below by the count the library itself reports
    log("per-kernel timing")
    saved_flag = trainer.use_graph
    trainer.use_graph = False
    prof_steps = 10
    trainer.step()
    barrier()
    if rank == 0:
        lib.siren_b200_profile_begin()
    for _ in range(prof_steps):
        trainer.step()
    barrier()
    trainer.use_graph = saved_flag
    if rank == 0:
        buf = ctypes.create_string_buffer(1 << 16)
        lib.siren_b200_profile_end(buf, len(buf))
        kernel_table = {}
        for ln in buf.value.decode().strip().splitlines():
            name, cnt, ms = ln.split()
            kernel_table[name] = {"launches": int(cnt), "avg_us": 1e3 * float(ms) / int(cnt),
                                  "us_per_step": 1e3 * float(ms) / prof_steps}
        # one entry per launch site of the library; the "adam" and "clip_grad" sites launch two kernels each
        launches_per_step = (sum(v["launches"] for v in kernel_table.values()) +
                             kernel_table.get("adam", {}).get("launches", 0) +
                             kernel_table.get("clip_grad", {}).get("launches", 0)) // prof_steps
        # Algorithmic work per launch (DESIGN.md section 3; bf16 planes of 256 features = 512 B per coordinate):
        #   mlp_fused_fwd  the whole forward: coordinates in (4 d), ONE fp16 stash plane per HIDDEN sine layer out (its
        #                  signed sine; N_HIDDEN x 512; the first layer's is recomputed from the coordinates), gt in, y + gy out
        #   mlp_fused_bwd  the dgrad chain from the loss gradient down: the stash planes of sine layers 1..N_HIDDEN in,
        #                  the adjoints of the same layers out (the weight-gradient kernel's operands)
        #   wgrad          adjoints of layers 1..N_HIDDEN in, stash planes of layers 1..N_HIDDEN-1 in (layer 0's operand is
        #                  built from the coordinates on chip)
        #   per-layer path (fp32-parity / SIREN_FUSED=0): hidden_fwd reads h (512) + writes h', c' (1024);
        #                  hidden_dgrad reads zbar, c (1024) + writes zbar' (512); fp32-parity doubles every plane
        pf = 1 if args.precision == "bf16" else 2
        abytes = {"hidden_fwd": 1536 * pf * n_local, "hidden_dgrad": 1536 * pf * n_local,
                  "wgrad": (1024 * pf * N_HIDDEN - (512 if args.precision == "bf16" else 0)) * n_local,
                  "mlp_fused_fwd": (N_HIDDEN * 512 + 4 * D_IN + 12 * D_OUT) * n_local,
                  "mlp_fused_bwd": (2 * N_HIDDEN * 512 + 4 * D_IN + 4 * D_OUT) * n_local}
        flops = {"hidden_fwd": HIDDEN_LAYER_FLOP * n_local, "hidden_dgrad": HIDDEN_LAYER_FLOP * n_local,
                 "wgrad": HIDDEN_LAYER_FLOP * n_local * N_HIDDEN,
                 "mlp_fused_fwd": HIDDEN_LAYER_FLOP * n_local * N_HIDDEN,
                 "mlp_fused_bwd": HIDDEN_LAYER_FLOP * n_local * N_HIDDEN}
        tc = {k: v for k, v in kernel_table.items() if k in flops}
        top = max(tc, key=lambda k: tc[k]["us_per_step"])
        sec = tc[top]["avg_us"] * 1e-6
        # dram__bytes_read.sum + dram__bytes_write.sum per launch of THIS build's kernels, from the committed
        # ncu --set full capture (profiles/r02_traffic.json, written by tools/ncu_summary.py); null when absent
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath) and args.precision == "bf16" and n_local == N_COORDS:
            traffic = json.load(open(tpath)).get(top)
        total_us = sum(v["us_per_step"] for v in kernel_table.values())
        # SURVEY 8(d): the roofline that bounds the path is the tensor cores (hidden layers are dense 256-wide
        # contractions); the HBM view of the same kernel is next to it
        roofline = {"bound": "tensor", "kernel": top, "achieved": flops[top] / sec / 1e12, "peak": pk["bf16_tflops"],
                    "unit": "TFLOP/s", "frac": flops[top] / sec / 1e12 / pk["bf16_tflops"], "traffic": traffic,
                    "algorithmic_flop_per_launch": flops[top], "peak_source": pk["source"] + " bf16_tflops (burst)",
                    "avg_us": tc[top]["avg_us"], "kernel_share_of_step": tc[top]["us_per_step"] / total_us,
                    "hbm": {"algorithmic_bytes_per_launch": abytes[top], "achieved_gbs": abytes[top] / sec / 1e9,
                            "peak_gbs": pk["hbm_gbs"], "frac": abytes[top] / sec / 1e9 / pk["hbm_gbs"]},
                    "per_kernel": {k: {"avg_us": v["avg_us"],
                                       "tensor_frac": flops[k] / (v["avg_us"] * 1e-6) / 1e12 / pk["bf16_tflops"],
                                       "hbm_frac": abytes[k] / (v["avg_us"] * 1e-6) / 1e9 / pk["hbm_gbs"]}
                                   for k, v in tc.items()},
                    "step_frac_of_peak": FLOP_PER_COORD * value / world / 1e12 / pk["bf16_tflops"],
                    "step_frac_of_sustained_peak": (FLOP_PER_COORD * value / world / 1e12 /
                                                    pk["bf16_tflops_sustained"]) if pk["bf16_tflops_sustained"] else None}

    # ---------------- strong scaling of cfg2 as BASELINE.json states it (N > 1) ----------------
    strong = None
    if world > 1 and args.scaling == "weak" and not args.quick:
        log("strong scaling: one 262144-coordinate batch over %d GPUs" % world)
        n_shard = (N_COORDS + world - 1) // world
        del trainer, model
        torch.cuda.empty_cache()
        m_s, tr_s = make_trainer(n_shard, args.precision)
        ch, gh = synthetic_batch(n_shard, rank, world, "strong")
        tr_s.coords.copy_(ch)
        tr_s.gt.copy_(gh)
        for _ in range(args.warmup):
            tr_s.step()
        ms_strong = timed_steps(tr_s, args.steps, barrier, dev, world)
        del tr_s, m_s
        # one GPU running the whole batch, in the same job on every rank (no communication), slowest rank counts
        m_1, tr_1 = make_trainer(N_COORDS, args.precision, use_dist=False)
        ch, gh = synthetic_batch(N_COORDS, 0, 1, "weak")
        tr_1.coords.copy_(ch)
        tr_1.gt.copy_(gh)
        for _ in range(args.warmup):
            tr_1.step()
        ms_one = timed_steps(tr_1, args.steps, barrier, dev, world)
        del tr_1, m_1
        strong = {"coords_per_step_global": N_COORDS, "coords_per_gpu": n_shard, "ms_per_step": ms_strong,
                  "value": N_COORDS / (ms_strong * 1e-3), "unit": "coords/s",
                  "one_gpu_ms_per_step": ms_one, "speedup_vs_one_gpu": ms_one / ms_strong,
                  "step_frac_of_peak": FLOP_PER_COORD * N_COORDS / (ms_strong * 1e-3) / world / 1e12 / pk["bf16_tflops"]}

    # ---------------- the other rows of SURVEY 8(d), N = 1 only ----------------
    parity_mode, configs, eager, cpu_baseline = None, None, None, None
    mri_blocks = []
    mri_step = []
    if rank == 0 and world == 1 and not args.quick:
        from tools import workloads
        del trainer, model
        torch.cuda.empty_cache()
        other = "fp32" if args.precision == "bf16" else "bf16"
        log("cfg2 in the %s mode" % other)
        m_p, tr_p = make_trainer(N_COORDS, other)
        tr_p.coords.copy_(coords_host)
        tr_p.gt.copy_(gt_host)
        for _ in range(5):
            tr_p.step()
        ms_p = timed_steps(tr_p, 50, barrier, dev, 1)
        parity_mode = {"precision_mode": other, "ms_per_step": ms_p, "value": N_COORDS / (ms_p * 1e-3), "unit": "coords/s",
                       "frac": FLOP_PER_COORD * N_COORDS / (ms_p * 1e-3) / 1e12 / pk["bf16_tflops"],
                       "tolerance": "rel-L2 <= 1e-4 vs the reference (tests/test_gpu_parity.py)" if other == "fp32"
                                    else "documented bf16 bound, DESIGN.md section 4"}
        del tr_p, m_p
        torch.cuda.empty_cache()
        configs = []
        for c in (1, 2, 3, 4, 5):
            for impl, prec, k in (("native", "bf16", 20), ("native", "fp32", 10), ("eager", "fp32", 3)):
                log("cfg%d %s %s" % (c, impl, prec))
                try:
                    r = workloads.run_config(c, impl, prec, steps=k, warmup=5 if impl == "native" else 2, dev=dev)
                    r["frac_of_peak"] = r["flop_per_coord"] * r["coords_per_sec"] / 1e12 / pk["bf16_tflops"]
                except Exception as e:      # a leg that fails must not take the headline line with it
                    r = {"config": workloads.NAMES[c], "impl": impl, "precision": prec, "error": repr(e)[:300]}
                configs.append(r)
            if c == 5:      # the same with the Fourier features built inside the kernels (siren_b200_forward_ff)
                for prec in ("bf16", "fp32"):
                    log("cfg5 lazy Fourier %s" % prec)
                    try:
                        r = workloads.run_config(5, "native", prec, steps=10, warmup=5, dev=dev, lazy_fourier=True)
                        r["frac_of_peak"] = r["flop_per_coord"] * r["coords_per_sec"] / 1e12 / pk["bf16_tflops"]
                    except Exception as e:
                        r = {"config": workloads.NAMES[5] + " (Fourier prologue in the kernels)", "impl": "native",
                             "precision": prec, "error": repr(e)[:300]}
                    configs.append(r)
            if c <= 4:      # the whole step as one graph of this library's kernels (what train_fast runs)
                for prec in ("bf16", "fp32"):
                    log("cfg%d trainer %s" % (c, prec))
                    try:
                        r = workloads.run_trainer_config(c, prec, dev=dev)
                        r["frac_of_peak"] = r["flop_per_coord"] * r["coords_per_sec"] / 1e12 / pk["bf16_tflops"]
                    except Exception as e:
                        r = {"config": workloads.NAMES[c], "impl": "native-trainer", "precision": prec, "error": repr(e)[:300]}
                    configs.append(r)
        # the MRI script's Fourier blocks (train_mri_neural_process_ddp.py:54-130), forward + MSE + backward at 8 tasks x
        # 65,536 coordinates in the bf16 mode: features built in the kernels / materialised by the reference's ops per step
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import probe_mri_blocks
            for F in (30, 128):
                for mode in ("lazy", "materialised"):
                    log("MRI block F=%d %s" % (F, mode))
                    mri_blocks.append(probe_mri_blocks.run(F, mode, steps=10))
        except Exception as e:
            mri_blocks.append({"error": repr(e)[:300]})
        # one GPU's share of the neural-process step around the hypo-network (cfg5: hypernetwork -> per-slice SIREN on
        # Fourier features -> data consistency -> losses -> backward into the hypernetwork; encoder skipped)
        try:
            import probe_mri_step
            for mode in ("native", "native-graph", "native-f", "reference"):
                log("MRI hypo-path step: %s" % mode)
                mri_step.append(probe_mri_step.run(mode, steps=10 if mode != "reference" else 3))
                torch.cuda.empty_cache()
        except Exception as e:
            mri_step.append({"error": repr(e)[:300]})
        e2 = [r for r in configs if r.get("impl") == "eager" and r["config"] == workloads.NAMES[2] and "error" not in r]
        if e2:
            eager = {"value": e2[0]["coords_per_sec"], "unit": "coords/s", "ms_per_step": e2[0]["ms_per_step"],
                     "what": "cfg2 through %s, eager PyTorch on this GPU, fp32, TF32 off, torch.optim.Adam" % e2[0]["model"],
                     "native_over_eager": value / e2[0]["coords_per_sec"]}

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("CPU baseline")
        threads = os.cpu_count() or 1
        sec, kind, what = cpu_reference_seconds(N_COORDS, 2, 1, threads)
        cpu_baseline = {"value": N_COORDS / sec, "unit": "coords/s", "cores": threads, "kind": kind,
                        "sample": "2 timed full 262144-coord steps after 1 warm-up; " + what,
                        "ms_per_step": sec * 1e3}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "coords/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "bf16x3",
            "data": "synthetic", "config": cfg,
            "mode": {"device": "cuda", "precision_mode": args.precision, "cuda_graph": not args.no_graph,
                     "operands": ("16-bit, fp32 accumulate: fp16 activations / weights in the forward, bf16 adjoints / "
                                  "weights in the backward, one fp16 stash plane per hidden layer (DESIGN.md section 2)")
                     if args.precision == "bf16" else "bf16 hi + lo split, 3 MMAs per product, fp32 accumulate and stash",
                     "timed_region_s": ms_step * args.steps * 1e-3, "allreduce": comm_used},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "kernels": kernel_table,
            "sustained": sustained, "parity_mode": parity_mode, "gpu_eager_baseline": eager, "strong": strong,
            "configs": configs, "mri_blocks": mri_blocks or None, "mri_step": mri_step or None, "loss_after": loss_after,
        }
        emit(line)
    sys.stdout.flush()
    if world > 1:
        # leave without tearing the communicator down: destroy_process_group() has been seen to hang
        # when collectives were captured into CUDA graphs; the processes are done anyway
        barrier()
        sys.stderr.flush()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
