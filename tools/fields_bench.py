"""Cost of writing the PDE loss in PyTorch on the decoder fields against the fused operator, on one GPU.

At bench.py's headline shape (B = 8 samples x 65 536 points, K = 6) and per mode, CUDA events around, after warm-up:
  1. fused   pde_residual forward + backward (one library call; the backward only scales cached gradients)
  2. fields  decoder_fields forward alone (dpn_decoder_jac_fwd)
  3. mse     decoder_fields + physics.residual_terms(nn.MSELoss()) + backward (dpn_decoder_jac_bwd recomputes pass 1)
  4. l1      the same with nn.L1Loss()
Each figure is the mean over --iters calls; the four are alternated per round so that clock and co-tenant drift hit all alike.
The card name, power limit and maximum SM clock are read in the same run.

    python tools/fields_bench.py [--modes f16x3,fp32] [--iters 10] [--rounds 3] [--out DIR]   -> DIR/fields_bench.json and stdout
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, iters):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--modes", default="f16x3,fp32")
    ap.add_argument("--B", type=int, default=8)
    ap.add_argument("--N", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fields_bench needs a GPU")
    import __graft_entry__
    __graft_entry__.build()
    from deepphysinet_b200 import functional as Fn, physics
    from deepphysinet_b200.config import PhysicsConsts
    from deepphysinet_b200.testing import random_decoder_weights

    consts = PhysicsConsts()
    W, pts = random_decoder_weights(B=a.B, N=a.N, seed=0)
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    Wl = Fn.DecoderWeights(*leaves)
    x, y, t, f, cd = pts["x"], pts["y"], pts["t"], pts["f"], pts["coord_data"]

    def clear():
        for l in leaves:
            l.grad = None

    def run(mode):
        def fused():
            clear()
            Fn.pde_residual(x, y, t, f, cd, Wl, consts=consts, mode=mode)[0].backward()

        def fields():
            with torch.no_grad():
                Fn.decoder_fields(x, y, t, cd, W, consts=consts, mode=mode)

        def loss_with(crit):
            def step():
                clear()
                o, jac = Fn.decoder_fields(x, y, t, cd, Wl, consts=consts, mode=mode)
                physics.residual_terms(o, jac, f, consts, crit).sum(1).mean().backward()
            return step
        return dict(fused=fused, fields=fields, mse=loss_with(nn.MSELoss()), l1=loss_with(nn.L1Loss()))

    res = dict(device=device_info(), B=a.B, N=a.N, iters=a.iters, rounds=a.rounds, modes={})
    for mode in a.modes.split(","):
        fns = run(mode)
        for fn in fns.values():                 # warm-up: module loads, workspace growth, allocator
            fn()
            fn()
        ms = {k: [] for k in fns}
        for _ in range(a.rounds):
            for k, fn in fns.items():
                ms[k].append(timed(fn, a.iters))
        best = {k: min(v) for k, v in ms.items()}
        res["modes"][mode] = dict(ms_per_call=ms, best_ms=best, mse_over_fused=best["mse"] / best["fused"],
                                  l1_over_fused=best["l1"] / best["fused"],
                                  mpts_per_s={k: a.B * a.N / v / 1e3 for k, v in best.items()})
        print("%-6s fused %.2f ms | fields fwd %.2f ms | fields+MSE+bwd %.2f ms (%.2fx) | fields+L1+bwd %.2f ms (%.2fx)" %
              (mode, best["fused"], best["fields"], best["mse"], best["mse"] / best["fused"], best["l1"], best["l1"] / best["fused"]))
    print(json.dumps(res["device"]))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "fields_bench.json"), "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
