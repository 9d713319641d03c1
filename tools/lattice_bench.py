"""Lattice inference on one B200: InterfacePhysics.predict_lattice against predict_grid.

  (a) bench.py's configs[3] workload - one sample, the 145 x 257 training grid, 48 hourly leads, cached generated weights -
      through predict_grid and predict_lattice, alternated in one run: ms per sweep, grid points/s, peak allocated memory.
  (b) the 4x refined domain (577 x 1025 nodes, 25 hourly leads) for B = 4 samples in one predict_lattice call.
  (c) kernel time of (a) and (b) from a separate torch.profiler run, and the achieved TFLOP/s on the 3.54 MFLOP/point of a
      values-only pass (BASELINE.md).
The coarse stacks hold 9 six-hourly slices (48 h) so that every lead of (a) lies inside them (bench.py's 5-slice stack covers
24 h; predict_grid samples NaN beyond it, predict_lattice refuses such a lattice).

    python tools/lattice_bench.py [--mode f16x3] [--iters 5] [--out DIR]   -> DIR/lattice_bench.json (and the text on stdout)
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

META_CFG = dict(name="TransformerNet", enc_in=2405, c_out=256, d_model=256, n_heads=8, e_layers=4, d_ff=256,
                dropout=0.5, activation="gelu", output_attention=False)
NET_CFG = dict(name="PhysicsNet", in_channels=192, hidden_channels=256, out_channels=1, token_num=159, learnable_token_num=256)
FLOP_PER_POINT = 3.54e6


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, iters):
    """Mean ms per call over `iters` calls (CUDA events) and the peak allocated memory of one call beyond what was live."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="f16x3")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of predict_grid / predict_lattice in (a)")
    ap.add_argument("--out", default=".", help="directory for lattice_bench.json (default: the current directory)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lattice_bench needs a GPU")
    import __graft_entry__ as G
    G.build()
    from deepphysinet_b200 import InterfacePhysics, functional as Fn, _native as N
    from deepphysinet_b200.config import DEFAULT_OBS_NORM
    dev = torch.device("cuda:0")
    obs = {k: dict(v, norm_type="mean_norm", use_norm=True) for k, v in DEFAULT_OBS_NORM.items()}
    torch.manual_seed(0)
    model = InterfacePhysics(META_CFG, NET_CFG, obs, None, dict(img_size=(145, 257), dx=27000, dy=27000)).to(dev)
    model.mode = args.mode
    g = torch.Generator().manual_seed(1)
    field = torch.randn(4, 159, 2405, generator=g).to(dev)
    fh = torch.full((4, 1, 1), 24.0 / 360.0).to(dev)
    coarse = torch.randn(4, 9, 37, 65, 6, generator=g).to(dev)
    with torch.no_grad():
        W4 = model.physics_net.decoder_weights(field, fh)
    W1 = Fn.DecoderWeights(*[(w[:1] if n in ("W1", "b1", "W2", "b2", "e") else w) for n, w in zip(Fn.DecoderWeights._fields, W4)])
    consts = model.consts(model._last_factor())
    res = {"device": device_info(), "mode": args.mode, "iters": args.iters}

    # (a) configs[3]: 145 x 257 x 48 hourly leads, one sample, cached weights
    model.pred_t_span = 48 * 3600.0
    leads = list(range(48))
    lat_a = Fn.Lattice.domain(consts, refine=1, st=3600.0, nt=48)
    npts_a = 145 * 257 * 48
    grid = lambda: model.predict_grid(field[:1], coarse[:1], fh[:1], leads, weights=W1)
    latt = lambda: model.predict_lattice(field[:1], coarse[:1], fh[:1], lat_a, weights=W1)
    same = torch.equal(grid(), latt()[0])
    rows = {"predict_grid": [], "predict_lattice": []}
    for _ in range(args.rounds):
        for name, fn in (("predict_grid", grid), ("predict_lattice", latt)):
            N.release_workspaces()
            torch.cuda.empty_cache()
            rows[name].append(timed(fn, args.iters))
    a = {}
    for name, r in rows.items():
        ms = sorted(x[0] for x in r)
        a[name] = {"ms_per_sweep_median": ms[len(ms) // 2], "ms_per_sweep_all": ms, "grid_points_per_s": npts_a / (ms[len(ms) // 2] * 1e-3),
                   "peak_allocated_MiB": max(x[1] for x in r) / 2 ** 20}
    a["outputs_bit_identical"] = same
    a["points"] = npts_a
    res["a_configs3_B1_145x257x48"] = a
    model.pred_t_span = 86400

    # (b) the 4x refined domain, 25 hourly leads, B = 4
    lat_b = Fn.Lattice.domain(consts, refine=4, st=3600.0, nt=25)
    npts_b = 4 * lat_b.nx * lat_b.ny * lat_b.nt
    big = lambda: model.predict_lattice(field, coarse, fh, lat_b, weights=W4)
    N.release_workspaces()
    torch.cuda.empty_cache()
    ms_b, peak_b = timed(big, max(1, args.iters // 2))
    res["b_refine4_B4_577x1025x25"] = {"ms_per_call": ms_b, "grid_points_per_s": npts_b / (ms_b * 1e-3), "points": npts_b,
                                       "peak_allocated_MiB": peak_b / 2 ** 20, "output_MiB": npts_b * 24 / 2 ** 20}

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "lattice_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    # (c) kernel time from a profiler run of its own
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for tag, fn, npts in (("a_predict_lattice", latt, npts_a), ("a_predict_grid", grid, npts_a), ("b_predict_lattice", big, npts_b)):
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                per[ev.key] = per.get(ev.key, 0.0) + ev.device_time_total / 1e3
        total = sum(per.values())
        top = sorted(per.items(), key=lambda kv: -kv[1])[:8]
        kern[tag] = {"kernel_ms_total": total, "TFLOP_per_s_on_3.54_MFLOP_per_point": npts * FLOP_PER_POINT / (total * 1e-3) / 1e12,
                     "top_kernels_ms": {k[:90]: v for k, v in top}}
    res["c_kernel_time"] = kern
    with open(os.path.join(args.out, "lattice_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
