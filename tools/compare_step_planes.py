#!/usr/bin/env python
"""Everything one siren_b200_forward_backward_mse call computes, dumped as .npy, and the comparison of two builds.

  python tools/compare_step_planes.py dump OUT [--root TREE]     run each case twice with TREE's library (default: this
                                                                 tree), write OUT/<case>/run<k>/<name>.npy
  python tools/compare_step_planes.py compare A B                 A, B: dump directories of two builds

Per case and run: y, gy, the loss accumulator, every dW / db, and the workspace's stash planes (signed sine of hidden
layers 1..L-1, fp16 bits) and adjoint planes (layers 1..L, bf16 bits), located as api.cu make_layout places them on the
fused bf16 path (d_in <= 4).  The one-kernel step fills y, gy and the planes in a fixed order: they must match bit for
bit.  The gradients and the loss are summed with atomic adds, so they are compared against the run-to-run spread of one
build (the two runs of each dump): the largest difference between the builds must stay within twice the larger of the
two builds' own spreads."""
import argparse
import os
import sys

import numpy as np

H = 256
W_MSE = 1.0 / 16384
CASES = {
    # name: d, n_hidden, o, tasks, per_task, n
    "cfg2": (2, 3, 1, 1, False, 262144),             # bench.py's headline shape (3 x 256, 262,144 coordinates)
    "pertask_2x20000_o2_nh4": (3, 4, 2, 2, True, 20000),
}


def plane_offsets(d, nh, tasks, per_task, n):
    """(stash {l: byte offset}, adjoint {l: byte offset}, bytes per plane) of the fused bf16 path (api.cu make_layout)."""
    Tw = tasks if per_task else 1
    n_pad = (n + 127) // 128 * 128
    plane = n_pad * tasks * H * 2
    off = [0]

    def take(nbytes):
        o = off[0]
        off[0] = (o + nbytes + 1023) // 1024 * 1024
        return o
    for _ in range(nh):
        take(Tw * H * H * 2)            # K-major weights
        take(Tw * H * H * 2)            # transposed weights
    take(Tw * H * 64 * 2)               # first layer as an MMA operand (unused for d <= 4)
    shared_c = take(plane)
    stash, adj = {}, {}
    for l in range(nh + 1):
        if 1 <= l < nh:
            stash[l] = take(plane)
        if l >= 1:
            adj[l] = take(plane)
    return stash, adj, plane


def dump(out, root):
    sys.path.insert(0, root)
    import torch
    from oracle import siren_oracle as so
    from siren_mri_b200 import _lib, functional as F
    lib = _lib.load()
    P = _lib.dptr
    print("library:", _lib.LIB_PATH)
    for case, (d, nh, o, T, per_task, n) in CASES.items():
        Ws, bs = so.make_params(d, H, nh, o, seed=11, tasks=T if per_task else 0)
        x = so.make_coords(T, n, d, seed=12)
        gt = np.random.default_rng(13).uniform(-1, 1, size=(T, n, o)).astype(np.float32)
        xd, gtd = torch.from_numpy(x).cuda(), torch.from_numpy(gt).cuda()
        Wd = [torch.from_numpy(w).cuda() for w in Ws]
        bd = [torch.from_numpy(b).cuda() for b in bs]
        desc = F._make_desc(xd, Wd, 30.0, "bf16", 0)
        nbytes = lib.siren_b200_workspace_bytes_ex(desc, 0)
        stash, adj, plane = plane_offsets(d, nh, T, per_task, n)
        for run in range(2):
            ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
            y = torch.zeros(T, n, o, device="cuda")
            gy = torch.zeros(T, n, o, device="cuda")
            grads = [torch.zeros(a.shape, device="cuda") for a in Ws + bs]
            loss4 = torch.zeros(4, device="cuda")
            torch.cuda.synchronize()
            _lib.check(lib.siren_b200_forward_backward_mse(
                desc, P(xd), _lib.ptr_array(Wd), _lib.ptr_array(bd), P(y), P(gtd), W_MSE, P(gy), P(loss4), P(ws), 0,
                _lib.ptr_array(grads[:len(Ws)]), _lib.ptr_array(grads[len(Ws):]), 0,
                torch.cuda.current_stream().cuda_stream), "forward_backward_mse")
            torch.cuda.synchronize()
            arrays = {"y": y, "gy": gy, "loss4": loss4}
            for i, g in enumerate(grads):
                arrays[("dW%d" if i < len(Ws) else "db%d") % (i % len(Ws))] = g
            for l, off in stash.items():
                arrays["stash%d" % l] = ws[off:off + plane].view(torch.int16)
            for l, off in adj.items():
                arrays["adj%d" % l] = ws[off:off + plane].view(torch.int16)
            dst = os.path.join(out, case, "run%d" % run)
            os.makedirs(dst, exist_ok=True)
            for name, t in arrays.items():
                np.save(os.path.join(dst, name + ".npy"), t.cpu().numpy())
        print("dumped", case)


def _load(root, case, run):
    dr = os.path.join(root, case, "run%d" % run)
    return {f[:-4]: np.load(os.path.join(dr, f)) for f in sorted(os.listdir(dr))}


def _maxdiff(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def compare(a_dir, b_dir):
    ok = True
    for case in sorted(os.listdir(a_dir)):
        a0, a1, b0, b1 = _load(a_dir, case, 0), _load(a_dir, case, 1), _load(b_dir, case, 0), _load(b_dir, case, 1)
        print("== %s" % case)
        for name in a0:
            bits = a0[name].tobytes() == b0[name].tobytes()
            if name.startswith(("y", "gy", "stash", "adj")):
                ok &= bits
                print("  %-8s %s" % (name, "bit-identical" if bits else "DIFFERS (%d elements)"
                                     % int((a0[name] != b0[name]).sum())))
            else:          # atomically summed: the builds' difference against each build's own run-to-run spread
                spread = max(_maxdiff(a1[name], a0[name]), _maxdiff(b1[name], b0[name]))
                cross = max(_maxdiff(b0[name], a0[name]), _maxdiff(b1[name], a1[name]))
                good = bits or cross <= 2 * spread
                ok &= good
                print("  %-8s %s  max|A-B| / max|A| %.2e, run-to-run spread %.2e" % (
                    name, "bit-identical" if bits else "within spread" if good else "OUTSIDE SPREAD", cross, spread))
    print("PASS" if ok else "FAIL")
    return ok


def main():
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    d = sub.add_parser("dump")
    d.add_argument("out")
    d.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    c = sub.add_parser("compare")
    c.add_argument("a")
    c.add_argument("b")
    args = ap.parse_args()
    if args.cmd == "dump":
        dump(args.out, os.path.abspath(args.root))
    else:
        sys.exit(0 if compare(args.a, args.b) else 1)


if __name__ == "__main__":
    main()
